"""Pin the C restatement (oracle/wrsn_oracle.c) against outputs of the reference itself.

The fixtures under tests/golden/ were produced by running the UNMODIFIED reference under the
oracle shims (oracle/gen_golden.py).  Integer / set / time quantities must match exactly, node and
charger energies to 1e-12 relative (observed: bit-exact), observations to 1e-9 absolute.
"""
import os

import numpy as np
import pytest

from oracle.ref_runner import reference_root
from oracle.wrsn_oracle import OracleWRSN
from tests.helpers import golden, golden_names, mc_dict_of, scenario_of

NETS = golden_names("net_")
EPS = golden_names("ep_")


def _close(a, b, rtol=1e-12, atol=0.0):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


@pytest.mark.parametrize("name", NETS)
def test_pure_network(name):
    g = golden(name)
    o = OracleWRSN(scenario_of(g), num_agent=0)
    o.start_network_only()
    N = int(g["N"])
    assert o.N == N
    # snapshots in time order
    prev = np.ones(N, np.uint8)
    deaths = []
    for key in g["snap_keys"]:
        t = float(str(key)[1:])
        o.run_until(t)
        nd = o.nodes()
        assert np.array_equal(nd["status"], g["%s_status" % key]), key
        assert np.array_equal(nd["level"], g["%s_level" % key]), key
        assert np.array_equal(o.targets_active(), g["%s_targets_active" % key]), key
        assert o.alive == int(g["%s_alive" % key]), key
        _close(nd["energy"], g["%s_energy" % key])
        _close(nd["cs"], g["%s_cs" % key])
        _close(nd["log_energy"], g["%s_log_energy" % key])
        died = np.nonzero((prev == 1) & (nd["status"] == 0))[0]
        prev = nd["status"].copy()
        deaths += [int(d) for d in died]
    assert deaths == [int(x) for x in g["deaths_node"]]
    o.run_until(float(g["end_time"]) + 0.75)   # gen_golden stops at end_time + 0.25 + 0.5
    assert o.netop_done()
    nd = o.nodes()
    _close(nd["energy"], g["final_energy"])
    assert abs(float(np.sum(nd["energy"])) - float(g["sum_energy_end"])) < 1e-6
    assert int(np.sum(o.targets_active() == 0)) == int(g["inactive_targets"])
    sg = o.static_graph()
    assert sorted(np.nonzero(sg["direct"])[0].tolist()) == sorted(int(x) for x in g["direct"])
    _close(o.consts()["frame"], g["frame"], rtol=0)


@pytest.mark.parametrize("name", EPS)
def test_episode(name):
    g = golden(name)
    M = int(g["num_agent"])
    S = int(g["map_size"])
    o = OracleWRSN(scenario_of(g), num_agent=M, mc=mc_dict_of(g), map_size=S)
    o.set_event_budget(3_000_000)
    full = {int(i): k for k, i in enumerate(g["full_state_idx"])}
    n = int(g["n"])
    for i in range(n):
        if i == 0:
            req = o.reset()
        else:
            fa = int(g["fed_agent"][i])
            req = o.step(fa, g["fed_action"][i])
        assert req["raw_agent_id"] == int(g["agent_id"][i]), (name, i)
        assert req["terminal"] == bool(g["terminal"][i]), (name, i)
        assert req["now"] == float(g["now"][i]), (name, i)
        nd = o.nodes()
        assert np.array_equal(nd["status"], g["status"][i]), (name, i)
        assert np.array_equal(nd["level"], g["level"][i]), (name, i)
        assert np.array_equal(o.targets_active(), g["targets_active"][i]), (name, i)
        assert o.alive == int(g["alive"][i])
        _close(nd["energy"], g["energy"][i])
        _close(nd["cs"], g["cs"][i])
        _close(nd["rr"], g["rr"][i], atol=1e-12)
        mc = o.mcs()
        _close(mc["loc"], g["mc_loc"][i])
        _close(mc["energy"], g["mc_energy"][i])
        assert np.array_equal(mc["status"], g["mc_status"][i])
        _close(mc["cpa"], g["mc_cpa"][i])
        assert np.array_equal(mc["type"], g["mc_type"][i])
        assert np.array_equal(mc["nconn"], g["mc_nconn"][i])
        _close(mc["excl"], g["excl"][i], rtol=1e-9, atol=1e-15)
        fm, _ = o.fitness()
        if np.isfinite(g["fitness_min"][i]):
            _close(fm, g["fitness_min"][i])
        if req["raw_agent_id"] >= 0:
            _close(req["action"], g["action"][i], rtol=0)
            if i > 0:
                _close(req["reward"], g["reward"][i], rtol=1e-9, atol=1e-18)
            _close(req["state"].reshape(4, -1).sum(1), g["chan_sum"][i], rtol=1e-10, atol=1e-12)
            if i in full:
                _close(req["state"], g["full_state"][full[i]], rtol=1e-10, atol=1e-13)
    _close(o.consts()["moving_time_max"], float(g["moving_time_max"]), rtol=0)
    _close(o.consts()["charging_time_max"], float(g["charging_time_max"]), rtol=0)
    _close(o.consts()["avg_nodes_agent"], float(g["avg_nodes_agent"]), rtol=1e-15)


@pytest.mark.skipif(reference_root() is None, reason="needs a checkout of the reference (set WRSN_REFERENCE_ROOT)")
def test_oracle_vs_live_reference_on_random_scenarios():
    """Beyond the frozen fixtures: the C restatement against the unmodified reference run here under the shims, two random
    synthetic scenarios with random actions (tests/fuzz_oracle_vs_reference.py is the long form: 44 configurations clean)."""
    import subprocess
    import sys
    from tests.helpers import REPO
    out = subprocess.run([sys.executable, os.path.join(REPO, "tests", "fuzz_oracle_vs_reference.py"), "--first-seed", "100",
                          "--count", "2", "--decisions", "6"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "0 failing configurations" in out.stdout
