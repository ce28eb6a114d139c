"""Parity checks shared by the CPU (host emulation) and GPU test files (TEST INFRASTRUCTURE).

Every check drives ``BatchedWRSN`` through the C ABI and compares with either the committed golden
fixtures (outputs of the unmodified reference, see oracle/gen_golden.py) or the C oracle run on the same
inputs.  Discrete quantities (agent ids, termination, status / level / coverage sets, event times) must be
identical.  Against the fixtures energies are compared at 1e-9 relative (spec: 1e-5); against the C oracle, which runs the
same arithmetic, every float the record and the request carry is compared bit for bit (``compare_row_with_oracle``) except
update_reward's outputs (reward, EXCL, detail[1]: 1e-9, DESIGN §5).  Observations, which go through exp(), at 1e-9
relative / 1e-9 absolute.
"""
import numpy as np
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, Scenario
from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict
from tests.helpers import golden, mc_dict_of

E_RTOL = 1e-9


def sc_from_golden(g):
    p = g["sc_par"]
    spe = dict(capacity=p[0], threshold=p[1], com_range=p[2], sen_range=p[3], prob_gp=p[4], package_size=p[5],
               er=p[6], et=p[7], efs=p[8], emp=p[9])
    return Scenario(nodes=g["sc_nodes"].reshape(-1, 2), targets=g["sc_targets"].reshape(-1, 2),
                    base_station=g["sc_bs"], node_phy_spe=spe, max_time=float(p[10]))


def _np(t):
    return t.detach().cpu().numpy().copy()


def check_pure_network(name, device, replicas=1):
    """runner/test_network.py logic (no chargers) against net_<scenario>.npz, every snapshot."""
    g = golden(name)
    env = BatchedWRSN(sc_from_golden(g), num_agent=0, num_envs=replicas, device=device)
    env.init_network(with_reward_process=False)
    bit_exact = 0
    for key in g["snap_keys"]:
        key = str(key)
        env.run_until(float(key[1:]))
        for b in range(replicas):
            assert np.array_equal(_np(env.view("status"))[b], g[key + "_status"]), (name, key)
            assert np.array_equal(_np(env.view("level"))[b].astype(np.int32), g[key + "_level"]), (name, key)
            assert np.array_equal(_np(env.targets_active())[b], g[key + "_targets_active"]), (name, key)
            assert int(_np(env.alive)[b]) == int(g[key + "_alive"]), (name, key)
            np.testing.assert_allclose(_np(env.view("energy"))[b], g[key + "_energy"], rtol=E_RTOL)
            np.testing.assert_allclose(_np(env.view("cs"))[b], g[key + "_cs"], rtol=E_RTOL)
            bit_exact += int(np.array_equal(_np(env.view("energy"))[b], g[key + "_energy"]))
    env.run_until(float(g["end_time"]) + 0.75)
    e = _np(env.view("energy"))[0]
    np.testing.assert_allclose(e, g["final_energy"], rtol=E_RTOL)
    assert abs(float(e.sum()) - float(g["sum_energy_end"])) < 1e-6
    assert int((_np(env.targets_active())[0] == 0).sum()) == int(g["inactive_targets"])
    assert float(_np(env.hdr("NET_ON"))[0]) == 0.0          # Network.operate has finished
    assert float(_np(env.hdr("ERR")).max()) == 0.0
    return bit_exact, len(g["snap_keys"]) * replicas


def check_episode(name, device, check_obs=False, replicas=1):
    """WRSN.reset/step with the fixture's injected actions against ep_<case>.npz, every decision."""
    g = golden(name)
    M, S = int(g["num_agent"]), int(g["map_size"])
    env = BatchedWRSN(sc_from_golden(g), num_agent=M, mc_type=mc_dict_of(g), num_envs=replicas, map_size=S, device=device)
    full = {int(i): k for k, i in enumerate(g["full_state_idx"])}
    n = int(g["n"])
    for i in range(n):
        if i == 0:
            req = env.reset()
        else:
            req = env.step(np.full(replicas, int(g["fed_agent"][i]), np.int32), np.tile(g["fed_action"][i], (replicas, 1)))
        fm = _np(env.get_network_fitness()[1])
        for b in range(replicas):
            tag = (name, i, b)
            aid = int(_np(req.agent_id)[b])
            assert aid == int(g["agent_id"][i]), tag
            assert int(_np(req.terminal)[b]) == int(g["terminal"][i]), tag
            assert float(_np(req.now)[b]) == float(g["now"][i]), tag
            assert int(_np(req.flags)[b]) == 0, tag
            assert np.array_equal(_np(env.view("status"))[b], g["status"][i]), tag
            assert np.array_equal(_np(env.view("level"))[b].astype(np.int32), g["level"][i]), tag
            assert np.array_equal(_np(env.targets_active())[b], g["targets_active"][i]), tag
            assert int(_np(env.alive)[b]) == int(g["alive"][i]), tag
            np.testing.assert_allclose(_np(env.view("energy"))[b], g["energy"][i], rtol=E_RTOL)
            np.testing.assert_allclose(_np(env.view("cs"))[b], g["cs"][i], rtol=E_RTOL)
            np.testing.assert_allclose(_np(env.view("rr"))[b], g["rr"][i], rtol=E_RTOL, atol=1e-12)
            np.testing.assert_allclose(_np(env.mc("X"))[b], g["mc_loc"][i][:, 0], rtol=1e-12)
            np.testing.assert_allclose(_np(env.mc("Y"))[b], g["mc_loc"][i][:, 1], rtol=1e-12)
            np.testing.assert_allclose(_np(env.mc("ENERGY"))[b], g["mc_energy"][i], rtol=E_RTOL)
            assert np.array_equal(_np(env.mc("STATUS"))[b].astype(np.uint8), g["mc_status"][i]), tag
            assert np.array_equal(_np(env.mc("TYPE"))[b].astype(np.uint8), g["mc_type"][i]), tag
            assert np.array_equal(_np(env.mc("NCONN"))[b].astype(np.int32), g["mc_nconn"][i]), tag
            np.testing.assert_allclose(_np(env.mc("CPA0"))[b], g["mc_cpa"][i][:, 0], rtol=1e-12)
            np.testing.assert_allclose(_np(env.mc("CPA1"))[b], g["mc_cpa"][i][:, 1], rtol=1e-12)
            np.testing.assert_allclose(_np(env.mc("CPA2"))[b], g["mc_cpa"][i][:, 2], rtol=1e-12)
            want_fm = float(g["fitness_min"][i])
            if np.isfinite(want_fm):
                np.testing.assert_allclose(fm[b], want_fm, rtol=1e-12, err_msg=str(tag))
            else:
                assert fm[b] == want_fm, (tag, fm[b], want_fm)
            np.testing.assert_allclose(_np(env.mc("EXCL"))[b], g["excl"][i], rtol=1e-9, atol=1e-15)
            if aid >= 0:
                assert np.array_equal(_np(req.action)[b], g["action"][i]), tag
                if i > 0:
                    np.testing.assert_allclose(float(_np(req.reward)[b]), float(g["reward"][i]), rtol=1e-9, atol=1e-18)
        if check_obs and int(g["agent_id"][i]) >= 0:
            obs = _np(env.get_state(dtype=torch.float64))
            for b in range(replicas):
                np.testing.assert_allclose(obs[b].reshape(4, -1).sum(1), g["chan_sum"][i], rtol=1e-9, atol=1e-9)
                if i in full:
                    np.testing.assert_allclose(obs[b], g["full_state"][full[i]], rtol=1e-9, atol=1e-12)
            if i in full:
                # float32 observation (what the policy networks consume; fp32 FFMA accumulation of fp64 exponentials):
                # within 1e-5 of the channel maximum, the tolerance the north star sets for floating-point state
                obs32 = _np(env.get_state(dtype=torch.float32)).astype(np.float64)
                ref = g["full_state"][full[i]]
                for ch in range(4):
                    tol = 1e-5 * max(float(np.abs(ref[ch]).max()), 1e-3)
                    assert float(np.abs(obs32[0][ch] - ref[ch]).max()) <= tol, (name, i, ch)
    return env.counters()


def _ordered(a):
    """float64 -> int64 keys whose order is the order of the values (-0.0 and +0.0 one apart): ulp distances."""
    i = np.ascontiguousarray(a, np.float64).view(np.int64).astype(np.int64)
    return np.where(i < 0, np.int64(-2 ** 63) - i, i)


def assert_bits(got, want, tag, what):
    """float64 arrays equal bit for bit (a NaN equals any NaN: the reference's ``inf - inf`` is whichever NaN the hardware makes);
    the failure names the worst ulp distance and where it is."""
    g = np.atleast_1d(np.ascontiguousarray(got, np.float64))
    w = np.atleast_1d(np.ascontiguousarray(want, np.float64))
    assert g.shape == w.shape, (tag, what, g.shape, w.shape)
    same = (g.view(np.int64) == w.view(np.int64)) | (np.isnan(g) & np.isnan(w))
    if not same.all():
        bad = np.nonzero(~same)[0]
        ulp = [abs(int(a) - int(b)) for a, b in zip(_ordered(g[bad]), _ordered(w[bad]))]
        k = int(np.argmax(ulp))
        raise AssertionError("%s: %s differs in %d of %d entries; worst %d ulp at [%d]: got %r, want %r"
                             % (tag, what, len(bad), g.size, ulp[k], bad[k], float(g[bad[k]]), float(w[bad[k]])))


_MC_BITS = ("X", "Y", "ENERGY", "CPA0", "CPA1", "CPA2")
_MC_INTS = (("TYPE", "type"), ("NCONN", "nconn"), ("STATUS", "status"))


def _request_views(env):
    """One host copy of everything check_vs_oracle compares, for all rows at once."""
    fit, fmin = env.get_network_fitness()
    v = {f: _np(env.view(f)) for f in ("status", "level", "energy", "cs", "rr", "mc", "hdr")}
    v["tact"], v["fit"], v["fmin"] = _np(env.targets_active()), _np(fit), _np(fmin)
    for f in ("agent_id", "terminal", "now", "action", "reward", "detail"):
        v["req_" + f] = _np(getattr(env.req, f))
    return v


def compare_row_with_oracle(env, v, b, o, r, prev_fit, k):
    """Row b of the host copy ``v`` (``_request_views``) against oracle ``o`` at its request ``r``, on the row's own columns.
    Exact: ids, termination, time, status / level / coverage sets, ALIVE, and bit for bit node energy / energyCS / energyRR, the
    chargers' X / Y / ENERGY / CPA0..2 / TYPE / NCONN / STATUS, per-target fitness and its minimum, the clipped action and the
    fitness term of the reward (detail[0] = the minimum now minus the minimum when the deciding charger was last stepped,
    ``prev_fit``).  To 1e-9: the reward, the
    exclusive reward EXCL and its term detail[1] (DESIGN §5: update_reward's reciprocal, table exponential and per-thread sums).
    Returns the oracle's fitness minimum."""
    E, tag = env.E, (b, k)
    aid = int(r["raw_agent_id"])
    assert int(v["req_agent_id"][b]) == aid, tag
    assert int(v["req_terminal"][b]) == int(r["terminal"]), tag
    assert float(v["req_now"][b]) == r["now"], tag
    nd = o.nodes()
    n = len(nd["energy"])
    assert np.array_equal(v["status"][b][:n], nd["status"]), tag
    assert np.array_equal(v["level"][b][:n].astype(np.int32), nd["level"]), tag
    assert np.array_equal(v["tact"][b][:o.T], o.targets_active()), tag
    assert float(v["hdr"][b][E["WRSN_H_ALIVE"]]) == float(o.alive), tag
    for f in ("energy", "cs", "rr"):
        assert_bits(v[f][b][:n], nd[f], tag, "node " + f)
    m, mcs = v["mc"][b][:o.M], o.mcs()
    want = dict(X=mcs["loc"][:, 0], Y=mcs["loc"][:, 1], ENERGY=mcs["energy"], CPA0=mcs["cpa"][:, 0], CPA1=mcs["cpa"][:, 1],
                CPA2=mcs["cpa"][:, 2])
    for f in _MC_BITS:
        assert_bits(m[:, E["WRSN_MC_" + f]], want[f], tag, "charger " + f)
    for f, g in _MC_INTS:
        assert np.array_equal(m[:, E["WRSN_MC_" + f]].astype(np.int64), mcs[g].astype(np.int64)), (tag, f)
    np.testing.assert_allclose(m[:, E["WRSN_MC_EXCL"]], mcs["excl"], rtol=1e-9, atol=1e-15, err_msg=str((tag, "EXCL")))
    omin, ofit = o.fitness()
    assert_bits(v["fit"][b][:o.T], ofit, tag, "per-target fitness")
    assert_bits(v["fmin"][b], omin, tag, "fitness minimum")
    if aid >= 0:
        assert_bits(v["req_action"][b], r["action"], tag, "clipped action")
        if k > 0:
            np.testing.assert_allclose(float(v["req_reward"][b]), r["reward"], rtol=1e-9, atol=1e-18, err_msg=str(tag))
            assert_bits(v["req_detail"][b][0], omin - prev_fit[aid], tag, "detail[0] (fitness term)")
            np.testing.assert_allclose(float(v["req_detail"][b][1]), mcs["excl"][aid] / o.consts()["avg_nodes_agent"], rtol=1e-9,
                                       atol=1e-18, err_msg=str((tag, "detail[1]")))
    return omin


def check_vs_oracle(scenarios, device, num_envs, steps, seed, num_agent=3, mc=None, check_obs=False, scale2=0.05,
                    map_size=100, scenario_index=None, controller=False, obs32=False, threads=0, rounds=0, probe=None, spread=0.0,
                    warm_up_time=100.0, before_step=None):
    """B environments with DIFFERENT action streams (and possibly different scenarios) vs B oracle runs (ladder L6), every
    row at every request as ``compare_row_with_oracle`` states.
    ``controller``: the actions are those of the reference's RandomController — the density map s0 + s1 - 10 s2 + s3 of the
    float32 observation, decoded ON THE DEVICE (wrsn_decode_density_map) — and the oracle is fed the decoded 3-vectors, so
    the simulation is compared on the trajectory the device controller drives (the decoder itself: tests/test_decode.py).
    ``obs32``: also the float32 raster against the oracle's state at 1e-5 of the channel maximum.
    ``probe(env, rows)``: called at every request with the boolean mask of the rows compared there (e.g. to count the
    requests that reached a regime the test is about).  ``spread``: the uniform actions are drawn from [-spread, 1 + spread]
    (before ``scale2``), so that the clipping of WRSN.step is exercised.  ``warm_up_time``: the simulated time before the first
    request, on both sides.  ``before_step(env, oracles, k, live, aid, act)``: called after the rows were compared at request k
    and before they are stepped with the actions ``act`` (e.g. to edit the same state in the engine and in the oracles)."""
    if isinstance(scenarios, Scenario):
        scenarios = [scenarios]
    env = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device, map_size=map_size,
                      scenario_index=scenario_index, threads=threads, step_rounds=rounds, warm_up_time=warm_up_time)
    sid = _np(env.scen_id)
    B = num_envs
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-spread, 1.0 + spread, size=(steps, B, 3))       # spread > 0: some components outside [0, 1] (clipped)
    acts[..., 2] *= scale2
    oracles = [OracleWRSN(scenario_from_dict(scenarios[sid[b]].to_dict()), num_agent=num_agent, mc=mc, map_size=map_size,
                          warm_up_time=warm_up_time) for b in range(B)]
    for o in oracles:
        o.set_event_budget(3_000_000)
    req = env.reset()
    oreq = [o.reset(want_state=check_obs or obs32) for o in oracles]
    prev_fit = [None] * B                                            # WRSN.reset :74-78: agents_prev_fitness
    fmin = [None] * B
    live = np.ones(B, bool)
    n_dec = 0
    for k in range(steps + 1):
        aid = _np(req.agent_id)
        v = _request_views(env)
        for b in range(B):
            if not live[b]:
                continue
            fmin[b] = compare_row_with_oracle(env, v, b, oracles[b], oreq[b], prev_fit[b], k)
            if k == 0:
                prev_fit[b] = [fmin[b]] * num_agent
            n_dec += int(oreq[b]["raw_agent_id"] >= 0)
        if probe is not None:
            probe(env, live.copy())
        if check_obs:
            obs = _np(env.get_state(dtype=torch.float64))
            for b in range(B):
                if live[b] and oreq[b]["raw_agent_id"] >= 0:
                    np.testing.assert_allclose(obs[b], oreq[b]["state"], rtol=1e-9, atol=1e-12)
        if obs32 or controller:
            o32 = env.get_state(dtype=torch.float32)
        if obs32:
            got = _np(o32).astype(np.float64)
            for b in range(B):
                if live[b] and oreq[b]["raw_agent_id"] >= 0:
                    ref = oreq[b]["state"]
                    for ch in range(4):
                        tol = 1e-5 * max(float(np.abs(ref[ch]).max()), 1e-3)
                        assert float(np.abs(got[b][ch] - ref[ch]).max()) <= tol, (b, k, ch)
        if k == steps:
            break
        live &= aid >= 0
        if not live.any():
            break
        mask = torch.as_tensor(live.astype(np.uint8))
        if controller:
            dm = o32[:, 0] + o32[:, 1] - 10.0 * o32[:, 2] + o32[:, 3]
            act_k = _np(env.density_map_to_action(dm.contiguous()))
            act_k[~live] = 0.0
        else:
            act_k = acts[k]
        if before_step is not None:
            before_step(env, oracles, k, live.copy(), aid, act_k)
        req = env.step(np.where(live, aid, -1).astype(np.int32), act_k, mask=mask)
        for b in range(B):
            if live[b]:
                if aid[b] >= 0:
                    prev_fit[b][int(aid[b])] = fmin[b]                # WRSN.step :299: the fitness before the step
                oreq[b] = oracles[b].step(int(aid[b]), act_k[b], want_state=check_obs or obs32)
    assert float(_np(env.hdr("ERR")).max()) == 0.0
    return n_dec, env.counters()


def check_network_after_operate_stopped(scenario, device, horizon, every=50.0, threads=0):
    """Nodes keep running after Network.operate has finished (alive == 0): levels stay stale, later deaths re-route
    through the stale levels (Node.find_receiver) — engine vs oracle far past the end of Network.operate."""
    env = BatchedWRSN(scenario, num_agent=0, num_envs=1, device=device, threads=threads)
    env.init_network(with_reward_process=False)
    o = OracleWRSN(scenario_from_dict(scenario.to_dict()), num_agent=0)
    o.start_network_only()
    t = 0.25
    while t < horizon:
        env.run_until(t)
        o.run_until(t)
        nd = o.nodes()
        assert np.array_equal(_np(env.view("status"))[0], nd["status"]), t
        assert np.array_equal(_np(env.view("level"))[0].astype(np.int32), nd["level"]), t
        np.testing.assert_allclose(_np(env.view("energy"))[0], nd["energy"], rtol=E_RTOL)
        np.testing.assert_allclose(_np(env.view("cs"))[0], nd["cs"], rtol=E_RTOL)
        t += every
    return env.counters(), int((nd["status"] == 0).sum())


def check_rollout_step(scenarios, device, num_envs, steps, seed, with_obs):
    """wrsn_rollout_step (step | reset-on-termination | observe in one call) == the same loop written with the
    individual entry points, over several episode boundaries."""
    rng = np.random.default_rng(seed)
    acts = rng.uniform(0.0, 1.0, size=(steps, num_envs, 3))
    acts[..., 2] *= 0.3                                  # long charges: episodes end inside the window
    a = BatchedWRSN(scenarios, num_agent=3, num_envs=num_envs, device=device)
    b = BatchedWRSN(scenarios, num_agent=3, num_envs=num_envs, device=device)
    a.reset(); b.reset()
    obs_a = torch.zeros((num_envs, 4, a.S, a.S), dtype=torch.float64, device=a.device) if with_obs else None
    resets = 0
    for k in range(steps):
        act = torch.as_tensor(acts[k], device=a.device)
        a.rollout_step(act, obs_a)
        aid = b.req.agent_id.clone()
        b.step(aid, act, mask=(aid >= 0))
        done = b.req.agent_id < 0
        resets += int(done.sum())
        b.reset(mask=done)
        for f in ("agent_id", "terminal", "now", "action"):
            assert torch.equal(getattr(a.req, f), getattr(b.req, f)), (k, f)
        ra, rb = _np(a.req.reward), _np(b.req.reward)
        assert np.array_equal(ra, rb, equal_nan=True), k
        assert torch.equal(a.state, b.state), k
        if with_obs:
            assert torch.equal(obs_a, b.get_state(dtype=torch.float64)) or bool((b.req.agent_id < 0).any()), k
    return resets


def _disable_batches(env):
    """TEST SWITCH hdr[OPT_NOBATCH]: every simulated second runs event by event (the path the batches must equal)."""
    env.hdr("OPT_NOBATCH")[:] = 1.0
    env.view("hdr", env._snap)[:, env.E["WRSN_H_OPT_NOBATCH"]] = 1.0


_STATE_FIELDS = ("hdr", "mc", "proc", "energy", "rr", "cs", "esend", "logc", "nbef", "naft", "level", "parent", "status",
                 "tact_words", "conn_words", "logtick", "ring")          # (the engine's scratch field is not state)


def _state_diff_but_switch(a, b):
    """'' when the two simulators' records are identical byte for byte (apart from the test switch and its counter),
    else a description of the first differing field."""
    ha, hb = a.view("hdr").clone(), b.view("hdr").clone()
    for f in ("OPT_NOBATCH", "NBATCH", "NSPLIT"):
        ha[:, a.E["WRSN_H_" + f]] = 0.0
        hb[:, b.E["WRSN_H_" + f]] = 0.0
    off = int(a._foff[a.E["WRSN_F_HDR"]]) + 8 * a.E["WRSN_H_LEN"]
    end = int(a._foff[a.E["WRSN_F_SCRATCH"]])            # the engine's scratch field (last in the record) is not state
    if torch.equal(ha.view(torch.int64), hb.view(torch.int64)) and torch.equal(a.state[:, off:end], b.state[:, off:end]):
        return ""
    for f in _STATE_FIELDS:
        x, y = (ha, hb) if f == "hdr" else (a.view(f), b.view(f))
        x, y = x.contiguous().view(torch.uint8).reshape(a.B, -1), y.contiguous().view(torch.uint8).reshape(a.B, -1)
        neq = x != y
        if bool(neq.any()):
            rows = torch.nonzero(neq.any(1)).flatten().tolist()
            cols = torch.nonzero(neq[rows[0]]).flatten().tolist()
            return "field %s envs %s byte columns %s" % (f, rows[:8], cols[:16])
    return "padding bytes differ"


def check_batches_equal_event_path(scenarios, device, num_envs, steps, seed, num_agent=3, scale2=0.3, threads=0, mc=None,
                                   probe=None, warm_up_time=100.0, before_step=None):
    """Whole-cycle batches (nodes_batch) leave EVERY byte of the environment record — node rows, event clock with its
    insertion counters, charger records — exactly as the event-by-event path does, over several episodes.  ``probe(env)``:
    called with the batched simulator after every step.  ``before_step(a, b, k, act)``: called before step k with both
    simulators and the actions (e.g. to edit the same state in both)."""
    rng = np.random.default_rng(seed)
    acts = rng.uniform(0.0, 1.0, size=(steps, num_envs, 3))
    acts[..., 2] *= scale2
    a = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device, threads=threads,
                    warm_up_time=warm_up_time)
    b = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device, threads=threads,
                    warm_up_time=warm_up_time)
    _disable_batches(b)
    a.reset(); b.reset()
    ends = 0
    for k in range(steps):
        if before_step is not None:
            before_step(a, b, k, acts[k])
        act = torch.as_tensor(acts[k], device=a.device)
        a.rollout_step(act); b.rollout_step(act)
        ends += int((a.req.now == a.warm_up_time).sum())           # rows that were just reset
        for f in ("agent_id", "terminal", "now", "action"):
            assert torch.equal(getattr(a.req, f), getattr(b.req, f)), (k, f)
        assert np.array_equal(_np(a.req.reward), _np(b.req.reward), equal_nan=True), k
        diff = _state_diff_but_switch(a, b)
        assert not diff, (k, diff)
        if probe is not None:
            probe(a)
    ca, cb = a.counters(), b.counters()
    # (the warm-up snapshot of `b` was simulated before the switch was set: its counter is not zero)
    assert ca["batched_ticks"] > cb["batched_ticks"] and ca["ticks"] == cb["ticks"] and ca["events"] == cb["events"]
    ca["batched_ticks"] -= cb["batched_ticks"]
    ca["episode_ends"] = ends
    return ca


def check_pure_network_batches(scenario, device, horizon, every):
    """Pure network (no chargers, no update_reward: four events per cycle) with and without batches."""
    a = BatchedWRSN(scenario, num_agent=0, num_envs=1, device=device)
    b = BatchedWRSN(scenario, num_agent=0, num_envs=1, device=device)
    a.init_network(with_reward_process=False); b.init_network(with_reward_process=False)
    b.hdr("OPT_NOBATCH")[:] = 1.0
    t = 0.25
    while t < horizon:
        a.run_until(t); b.run_until(t)
        diff = _state_diff_but_switch(a, b)
        assert not diff, (t, diff)
        t += every
    return a.counters()


def _toy_policy(salt, clock, use_obs):
    """Deterministic stand-in for IPPO.get_action: a 3-vector action and a 'log-probability' that depend on the agent, a
    per-environment salt, the simulation time of the request and (``use_obs``) the observation only."""
    def policy(agent_id, obs):
        now = clock().to(torch.float64)
        s = torch.as_tensor(salt, dtype=torch.float64, device=now.device)
        a = agent_id.to(torch.float64)
        m0 = m1 = torch.zeros_like(now)
        if use_obs:
            m = obs.to(torch.float64).mean(dim=(2, 3))                              # [B, 4]
            m0, m1 = 1e3 * m[:, 0], 7e2 * m[:, 1]
        u = torch.stack((torch.frac(m0 + 0.37 * s + 0.11 * a + 0.013 * now), torch.frac(m1 + 0.53 * s + 0.29 * a + 0.007 * now),
                         0.25 * torch.frac(0.71 * s + 0.0031 * now)), dim=1)
        return u.to(torch.float32), (torch.sin(now) + 0.01 * a).to(torch.float32)
    return policy


def check_ippo_rollout(scenarios, device, num_envs, steps, gamma=0.99, lam=0.95, with_obs=True, windows=1):
    """IPPORollout (batched, linked record) == the reference's roll_out loop (IPPO.py:128-155) written against the
    single-environment façade, environment by environment: the same transitions in the same order for every agent,
    and cal_rt_adv == the reference's recursion over every (episode, agent) list.  ``with_obs=False``: no observations
    (the host emulation has no raster); the critic is then a function of the requests' simulation times.  ``windows`` > 1: the same
    steps collected in several windows with ``keep_open`` — no transition may be lost at a window boundary."""
    from multi_agent_rl_wrsn_b200 import WRSN
    from multi_agent_rl_wrsn_b200.controllers import IPPORollout

    class _NoObsWRSN(WRSN):
        def get_state(self, agent_id):
            return None
    M = 3
    env = BatchedWRSN(scenarios, num_agent=M, num_envs=num_envs, device=device)
    env.reset()
    ro = IPPORollout(env, steps // windows, action_shape=(3,), obs_dtype=torch.float64, with_obs=with_obs, keep_open=windows > 1)
    salt = np.arange(num_envs)
    value_fn = lambda s: (s[:, 0].mean(dim=(1, 2)) * 50.0 + s[:, 1].mean(dim=(1, 2))).to(torch.float32)
    value_t = lambda t: torch.cos(0.01 * torch.as_tensor(t, dtype=torch.float64)).to(torch.float32)

    def per_agent_of_window():
        res = []
        for i in range(M):
            bt = ro.batch(i, states=False, next_states=False)
            kw = {} if with_obs else dict(values=value_t(bt["prev_time"]), next_values=value_t(bt["time"]))
            returns, advantages, values, bt = ro.cal_rt_adv(i, value_fn, gamma, lam, **kw)
            if with_obs:
                bt["next_states"] = ro.obs[bt["t"], bt["b"]]
            res.append((returns, advantages, values, bt))
        return res

    n_tr = episodes = 0
    if windows > 1:                                           # window by window; rows of one environment stay in time order
        parts = []
        for w in range(windows):
            ro.carry_over()
            ro.collect(_toy_policy(salt, lambda: env.req.now, with_obs))
            parts.append(per_agent_of_window())
        keys_cat = ("actions", "log_probs", "rewards", "prev_time", "time", "b") + (("states", "next_states") if with_obs else ())
        merged = []
        for i in range(M):
            bt = {k: torch.cat([p[i][3][k] for p in parts]) for k in keys_cat}
            merged.append(tuple(torch.cat([p[i][j] for p in parts]) for j in range(3)) + (bt,))
    else:
        ro.collect(_toy_policy(salt, lambda: env.req.now, with_obs))
    for tf in ((None,) if windows > 1 else (None, 1.0)):      # the reference's all-False terminals, and a live recursion
        ro.terminal_factor = tf
        per_agent = merged if windows > 1 else per_agent_of_window()
        for b in range(num_envs):
            single = (WRSN if with_obs else _NoObsWRSN)(scenarios[b % len(scenarios)], None, M, device=device)
            pol = _toy_policy(salt[b:b + 1], lambda: single._b.req.now, with_obs)
            keys = ("states", "actions", "log_probs", "rewards", "next_states", "prev_time", "time")
            rec = [dict({k: [] for k in keys}, adv=[], ret=[]) for _ in range(M)]
            done = 0
            first = True
            while done < steps:
                if not first:
                    episodes += 1
                first = False
                request = single.reset()
                lists = [{k: [] for k in keys} for _ in range(M)]
                pre, asked = [None] * M, [None] * M
                while done < steps:
                    aid = request["agent_id"]
                    x, lp = pol(torch.tensor([aid], dtype=torch.int32, device=device),
                                torch.as_tensor(request["state"], device=device)[None] if with_obs else None)
                    pre[aid], asked[aid] = float(lp[0]), single.env.now
                    request = single.step(aid, x[0].cpu().numpy().astype(np.float64))
                    done += 1
                    if request["terminal"]:
                        break
                    aid = request["agent_id"]
                    if pre[aid] is None:
                        continue
                    L = lists[aid]
                    L["states"].append(request["prev_state"]); L["actions"].append(request["input_action"])
                    L["next_states"].append(request["state"]); L["rewards"].append(request["reward"]); L["log_probs"].append(pre[aid])
                    L["prev_time"].append(asked[aid]); L["time"].append(single.env.now)
                for i in range(M):                             # IPPO.cal_rt_adv :71-83 on this episode's list
                    L = lists[i]
                    if not L["rewards"]:
                        continue
                    if with_obs:
                        v = value_fn(torch.as_tensor(np.array(L["states"])))
                        nv = value_fn(torch.as_tensor(np.array(L["next_states"])))
                    else:
                        v, nv = value_t(L["prev_time"]), value_t(L["time"])
                    r = torch.tensor(L["rewards"], dtype=torch.float32)
                    term = 0.0 if tf is None else tf
                    adv = torch.zeros_like(r)
                    last = 0.0
                    for t in reversed(range(len(r))):
                        delta = r[t] + gamma * nv[t] * term - v[t]
                        last = delta + gamma * lam * term * last
                        adv[t] = last
                    for k in keys:
                        rec[i][k].extend(L[k])
                    rec[i]["adv"].extend(adv.tolist()); rec[i]["ret"].extend((adv + v).tolist())
            for i in range(M):
                returns, advantages, values, bt = per_agent[i]
                sel = torch.sort((bt["b"] == b).nonzero()[:, 0]).values        # (several windows: already window-major = time order)
                assert len(sel) == len(rec[i]["rewards"]), (b, i, len(sel), len(rec[i]["rewards"]))
                if not len(sel):
                    continue
                n_tr += len(sel)
                g = lambda k: bt[k][sel].cpu().numpy()
                if with_obs:
                    assert np.allclose(g("states"), np.array(rec[i]["states"]), rtol=1e-9, atol=1e-12), (b, i)
                    assert np.allclose(g("next_states"), np.array(rec[i]["next_states"]), rtol=1e-9, atol=1e-12), (b, i)
                assert np.array_equal(g("prev_time"), np.array(rec[i]["prev_time"])), (b, i)
                assert np.array_equal(g("time"), np.array(rec[i]["time"])), (b, i)
                assert np.allclose(g("actions"), np.array(rec[i]["actions"]), rtol=0, atol=1e-7), (b, i)
                assert np.allclose(g("log_probs"), np.array(rec[i]["log_probs"]), rtol=1e-6), (b, i)
                assert np.allclose(g("rewards"), np.array(rec[i]["rewards"], np.float32), rtol=1e-6, atol=1e-9), (b, i)
                assert np.allclose(advantages[sel].cpu().numpy(), np.array(rec[i]["adv"]), rtol=1e-4, atol=1e-6), (b, i)
                assert np.allclose(returns[sel].cpu().numpy(), np.array(rec[i]["ret"]), rtol=1e-4, atol=1e-6), (b, i)
    return n_tr, episodes


def check_charge_kernel(scenarios, device, num_envs, steps, seed, num_agent=3, mc=None, probe=None):
    """wrsn_k_charge (dense node x charger charging model, one warp per environment) == the reference's statements
    (oracle.wrsn_oracle.charge_rates_reference), bit for bit, on states reached by a rollout whose actions send the chargers to
    node positions (several nodes within range), with all chargers and with a random subset selected.  ``probe(env)``: called
    at every step whose rates are checked."""
    from oracle.wrsn_oracle import charge_rates_reference
    env = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device)
    sid = _np(env.scen_id)
    rng = np.random.default_rng(seed)
    env.reset()
    n_pairs = n_exact = n_rows = 0
    for k in range(steps):
        act = np.zeros((num_envs, 3))
        for b in range(num_envs):
            st = env.statics[sid[b]]
            par, sc = st["par"], env.scenarios[sid[b]]
            n = rng.integers(sc.N)
            xy = sc.nodes[n] + rng.normal(0.0, 8.0, 2)                      # a few metres off a node
            act[b, 0] = np.clip((xy[0] - par["F0"]) / (par["F1"] - par["F0"]), 0, 1)
            act[b, 1] = np.clip((xy[1] - par["F2"]) / (par["F3"] - par["F2"]), 0, 1)
            act[b, 2] = rng.uniform(0, 0.02)
        env.rollout_step(torch.as_tensor(act, device=env.device))
        if k % 3:
            continue
        if probe is not None:
            probe(env)
        for sel in (None, rng.integers(0, 2, size=(num_envs, num_agent)).astype(np.uint8)):
            node_rate, mc_rate = env.charge_rates(None if sel is None else torch.as_tensor(sel, device=env.device))
            node_rate, mc_rate = _np(node_rate), _np(mc_rate)
            status, mx, my = _np(env.view("status")), _np(env.mc("X")), _np(env.mc("Y"))
            for b in range(num_envs):
                mcp = env.mc_type
                rr, cr = charge_rates_reference(env.scenarios[sid[b]].nodes, status[b], np.stack([mx[b], my[b]], 1),
                                                np.ones(num_agent) if sel is None else sel[b],
                                                mcp["charging_range"], mcp["alpha"], mcp["beta"])
                # same connected sets; rates to the last bits (1e-14: a host whose libm / BLAS rounds differently must not fail
                # the run, a wrong model would be off by orders of magnitude); exact matches are counted and reported
                assert np.array_equal(node_rate[b] != 0, rr != 0), (k, b)
                assert np.array_equal(mc_rate[b] != 0, cr != 0), (k, b)
                np.testing.assert_allclose(node_rate[b], rr, rtol=1e-14, atol=0, err_msg=str((k, b)))
                np.testing.assert_allclose(mc_rate[b], cr, rtol=1e-14, atol=0, err_msg=str((k, b)))
                n_pairs += int((rr != 0).sum())
                n_exact += int(np.array_equal(node_rate[b], rr) and np.array_equal(mc_rate[b], cr))
                n_rows += 1
    print("charge kernel: %d connected pairs, %d / %d rows bit-identical" % (n_pairs, n_exact, n_rows))
    return n_pairs


def check_budget_equals_unbudgeted(scenarios, device, num_envs, calls, seed, budget, num_agent=3, scale2=0.3, threads=0, rounds=0,
                                   mc=None, probe=None, launch_probe=None):
    """A step budget (wrsn_dims.step_budget) only cuts a WRSN.step into several launches: every request an environment hands
    out — agent, time, reward, termination, clipped action — and every byte of its record at that moment are those of the
    unbudgeted run answered with the same actions.  Returns how many interrupted launches it took.  ``probe(env)``: called with
    the unbudgeted simulator after every step; ``launch_probe(env)``: with the budgeted one after every launch."""
    rng = np.random.default_rng(seed)
    acts = rng.uniform(0.0, 1.0, size=(calls, num_envs, 3))
    acts[..., 2] *= scale2
    a = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device, threads=threads)
    b = BatchedWRSN(scenarios, num_agent=num_agent, mc_type=mc, num_envs=num_envs, device=device, threads=threads,
                    step_budget=budget, step_rounds=rounds)
    end = int(a._foff[a.E["WRSN_F_SCRATCH"]])            # the engine's scratch field (last in the record) is not state
    hdr0 = int(a._foff[a.E["WRSN_F_HDR"]])
    skip = [hdr0 + 8 * a.E["WRSN_H_" + f] for f in ("NRESUME", "NBATCH")]   # (a split step may run a short batch event by event)

    def rows(env):
        st = env.state[:, :end].clone()
        for o in skip:
            st[:, o:o + 8] = 0
        return st.cpu()

    fields = ("agent_id", "terminal", "now", "action", "reward", "detail", "flags")
    a.reset(); b.reset()
    rec = []
    for k in range(calls):
        a.rollout_step(torch.as_tensor(acts[k], device=a.device))
        rec.append(({f: _np(getattr(a.req, f)) for f in fields}, rows(a)))
        assert not bool((a.req.agent_id == -4).any())
        if probe is not None:
            probe(a)
    count = np.zeros(num_envs, np.int64)
    interrupted = launches = 0
    while int(count.min()) < calls and launches < 400 * calls:
        cur = np.minimum(count, calls - 1)
        act = torch.as_tensor(acts[cur, np.arange(num_envs)], device=b.device)
        b.rollout_step(act)
        launches += 1
        if launch_probe is not None:
            launch_probe(b)
        aid = _np(b.req.agent_id)
        st = rows(b)
        got = {f: _np(getattr(b.req, f)) for f in fields}
        for e in range(num_envs):
            if aid[e] == -4:
                interrupted += 1
                continue
            if count[e] >= calls:
                continue
            want, wst = rec[count[e]]
            for f in fields:
                assert np.array_equal(got[f][e], want[f][e], equal_nan=True), (e, int(count[e]), f, got[f][e], want[f][e])
            assert torch.equal(st[e], wst[e]), (e, int(count[e]), "state record differs")
            count[e] += 1
    assert int(count.min()) >= calls, "budgeted run did not finish"
    return interrupted


def check_tick_kernels(name, device, t_from, t_to):
    """Ladder L1 / L2: the standalone per-tick kernels (wrsn_k_drain k+0.5, wrsn_k_bookkeep k+1.0, wrsn_k_bfs k+1.1) applied by
    hand, tick after tick, to a state dumped from a pure-network run of a shipped scenario — against the oracle advanced
    through the same ticks, across the death tick.  Returns the number of deaths seen."""
    g = golden(name)
    sc = sc_from_golden(g)
    env = BatchedWRSN(sc, num_agent=0, num_envs=1, device=device)
    env.init_network(with_reward_process=False)
    o = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=0)
    o.start_network_only()
    env.run_until(t_from + 0.25)                     # second t_from: connectivity at +0.1 done, drain at +0.5 next
    o.run_until(t_from + 0.25)
    dead0 = int((o.nodes()["status"] == 0).sum())

    def same(tag, with_levels):
        nd = o.nodes()
        assert np.array_equal(_np(env.view("status"))[0], nd["status"]), tag
        np.testing.assert_allclose(_np(env.view("energy"))[0], nd["energy"], rtol=E_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(_np(env.view("cs"))[0], nd["cs"], rtol=E_RTOL, err_msg=str(tag))
        if with_levels:
            assert np.array_equal(_np(env.view("level"))[0].astype(np.int32), nd["level"]), tag
            assert np.array_equal(_np(env.targets_active())[0], o.targets_active()), tag
            assert int(_np(env.alive)[0]) == int(o.alive), tag

    for k in range(int(t_from), int(t_to)):
        env.kernel("drain"); o.run_until(k + 0.75); same((k, "drain"), False)
        env.kernel("bookkeep"); o.run_until(k + 1.05); same((k, "bookkeep"), False)
        if float(_np(env.hdr("BFS_DIRTY"))[0]) != 0.0:
            env.kernel("bfs")
        o.run_until(k + 1.25); same((k, "bfs"), True)
    return int((o.nodes()["status"] == 0).sum()) - dead0


def reward_tick_reference(energy, cs, status, thr, cap, eps, mc_xy, mc_charging, conn, xy, alpha, beta):
    """WRSN.update_reward (rl_env/WRSN.py:100-127), one tick, restated with numpy on plain arrays: the increments of
    agents_exclusive_reward."""
    pr = np.where(status != 0, cs / (energy - thr + eps), 0.0)
    mean, std = np.mean(pr), np.std(pr)
    if std == 0:
        std = eps
    pr = np.exp((pr - mean) / std)
    tot = np.sum(pr)
    if tot == 0:
        tot = eps
    pr = pr / tot
    out = np.zeros(len(mc_xy))
    for a in range(len(mc_xy)):
        if not mc_charging[a]:
            continue
        inc = 0.0
        for n in conn[a]:
            if status[n] == 1:
                d = float(np.sqrt((xy[n, 0] - mc_xy[a, 0]) ** 2 + (xy[n, 1] - mc_xy[a, 1]) ** 2))
                rate = alpha / (d + beta) ** 2
                e_no = min(energy[n] - cs[n], thr)
                e_with = max(energy[n] - cs[n] + rate, cap)
                inc += pr[n] * (e_with - e_no) / (alpha / beta ** 2)
        out[a] = inc
    return out


def check_reward_kernel(scenarios, device, num_envs, steps, seed, num_agent=3):
    """wrsn_k_reward (one WRSN.update_reward tick: softmax of z-scored priorities + incentive sums, reciprocal / table-exp
    arithmetic) against the numpy restatement of the reference's statements on states reached by a rollout that parks the
    chargers next to nodes.  Returns the number of (charger, tick) increments compared that were non-zero."""
    env = BatchedWRSN(scenarios, num_agent=num_agent, num_envs=num_envs, device=device)
    sid = _np(env.scen_id)
    rng = np.random.default_rng(seed)
    env.reset()
    n_nonzero = 0
    for k in range(steps):
        act = np.zeros((num_envs, 3))
        for b in range(num_envs):
            st = env.statics[sid[b]]
            par, sc = st["par"], env.scenarios[sid[b]]
            xy = sc.nodes[rng.integers(sc.N)] + rng.normal(0.0, 6.0, 2)
            act[b, 0] = np.clip((xy[0] - par["F0"]) / (par["F1"] - par["F0"]), 0, 1)
            act[b, 1] = np.clip((xy[1] - par["F2"]) / (par["F3"] - par["F2"]), 0, 1)
            act[b, 2] = rng.uniform(0.02, 0.1)
        env.rollout_step(torch.as_tensor(act, device=env.device))
        before = _np(env.mc("EXCL"))
        energy, cs, status = _np(env.view("energy")), _np(env.view("cs")), _np(env.view("status"))
        mx, my, typ, mst = _np(env.mc("X")), _np(env.mc("Y")), _np(env.mc("TYPE")), _np(env.mc("STATUS"))
        conn = _np(env.view("conn_words")).astype(np.int64) & 0xFFFFFFFF
        env.kernel("reward")
        after = _np(env.mc("EXCL"))
        for b in range(num_envs):
            par = env.statics[sid[b]]["par"]
            sets = [[n for n in range(env.N) if (conn[b, a, n >> 5] >> (n & 31)) & 1] for a in range(num_agent)]
            ref = reward_tick_reference(energy[b], cs[b], status[b], par["THR"], par["CAP"], par["EPSENV"],
                                        np.stack([mx[b], my[b]], 1), (typ[b] != 0) & (mst[b] != 0), sets,
                                        np.asarray(env.scenarios[sid[b]].nodes, np.float64), par["MC_ALPHA"], par["MC_BETA"])
            np.testing.assert_allclose(after[b] - before[b], ref, rtol=1e-9, atol=1e-12 * max(1.0, float(np.abs(before[b]).max())),
                                       err_msg=str((k, b)))
            n_nonzero += int((ref != 0).sum())
    return n_nonzero


def check_sharded_equals_unsharded(scenarios, device, num_envs, steps, seed, world=2, num_agent=3, budget=0, rounds=0):
    """Environments shard by index: the records of `world` simulators holding contiguous blocks of the environments are, byte
    for byte, the blocks of ONE simulator holding all of them (same scenario assignment, same actions)."""
    from multi_agent_rl_wrsn_b200.sharding import shard_range, shard_scenario_index
    rng = np.random.default_rng(seed)
    acts = rng.uniform(0.0, 1.0, size=(steps, num_envs, 3))
    acts[..., 2] *= 0.1
    whole = BatchedWRSN(scenarios, num_agent=num_agent, num_envs=num_envs, device=device, step_budget=budget, step_rounds=rounds,
                        scenario_index=shard_scenario_index(num_envs, len(scenarios), 0, 1))
    parts = []
    for r in range(world):
        lo, hi = shard_range(num_envs, r, world)
        parts.append((lo, hi, BatchedWRSN(scenarios, num_agent=num_agent, num_envs=hi - lo, device=device, step_budget=budget,
                                          step_rounds=rounds, scenario_index=shard_scenario_index(num_envs, len(scenarios), r, world))))
    whole.reset()
    for _, _, p in parts:
        p.reset()
    end = int(whole._foff[whole.E["WRSN_F_SCRATCH"]])
    for k in range(steps):
        whole.rollout_step(torch.as_tensor(acts[k], device=whole.device))
        for lo, hi, p in parts:
            p.rollout_step(torch.as_tensor(acts[k, lo:hi], device=p.device))
            assert torch.equal(p.state[:, :end], whole.state[lo:hi, :end]), (k, lo)
            for f in ("agent_id", "terminal", "now", "action", "reward"):
                assert np.array_equal(_np(getattr(p.req, f)), _np(getattr(whole.req, f))[lo:hi], equal_nan=True), (k, lo, f)
    return whole.counters()
