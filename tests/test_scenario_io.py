"""Scenario I/O (SURVEY §8 f3): the reference's YAML schema, the bacgiang fix-up switch, the static graph of all nine shipped
scenarios against the oracle's (ladder L0).  The shipped YAML files are not part of this repository: the tests that read
them run where a checkout of the reference is found (oracle/ref_runner.py: $WRSN_REFERENCE_ROOT) and are skipped elsewhere.
The five shipped scenarios stored as arrays in tests/golden/net_*.npz are checked without one."""
import glob
import os

import numpy as np
import pytest
import yaml

from multi_agent_rl_wrsn_b200 import Scenario, synthetic
from multi_agent_rl_wrsn_b200.scenario import SHIPPED_MAX_TIME, build_static, load_mc_type
from oracle.ref_runner import reference_root
from tests.helpers import golden, golden_names, scenario_of

SHIPPED = os.path.join(reference_root() or "", "physical_env", "network", "network_scenarios")
needs_reference = pytest.mark.skipif(reference_root() is None, reason="needs a checkout of the reference (set WRSN_REFERENCE_ROOT)")


def test_yaml_round_trip(tmp_path):
    sc = synthetic(num_nodes=30, num_targets=40, seed=5)
    p = tmp_path / "s.yaml"
    sc.save_yaml(p)
    back = Scenario.load_yaml(p)
    assert np.array_equal(back.nodes, sc.nodes) and np.array_equal(back.targets, sc.targets)
    assert back.max_time == sc.max_time and back.node_phy_spe == sc.node_phy_spe
    d = yaml.safe_load(open(p))
    assert set(d) == {"node_phy_spe", "seed", "max_time", "base_station", "nodes", "targets"}      # NetworkIO.py:19-34


def test_missing_max_time_raises_like_the_reference_unless_fixed_up():
    d = synthetic(num_nodes=20, num_targets=20, seed=1).to_dict()
    del d["max_time"]
    with pytest.raises(KeyError):
        Scenario.from_dict(d)                                          # NetworkIO.py:34
    assert Scenario.from_dict(d, default_max_time=SHIPPED_MAX_TIME).max_time == SHIPPED_MAX_TIME


@pytest.mark.parametrize("name", golden_names("net_"))
def test_stored_shipped_scenarios_match_the_oracle_graph(name):
    """L0 without a checkout: the shipped scenarios stored as arrays in the reference's pure-network fixtures.  The static graph
    built for the engine equals the oracle's, and its base-station-direct set equals the one the reference itself reported."""
    from oracle.wrsn_oracle import OracleWRSN
    g = golden(name)
    q = g["sc_par"]
    spe = dict(capacity=q[0], threshold=q[1], com_range=q[2], sen_range=q[3], prob_gp=q[4], package_size=q[5],
               er=q[6], et=q[7], efs=q[8], emp=q[9])
    sc = Scenario(nodes=g["sc_nodes"].reshape(-1, 2), targets=g["sc_targets"].reshape(-1, 2), base_station=g["sc_bs"],
                  node_phy_spe=spe, max_time=float(q[10]), name=name)
    st = build_static(sc, load_mc_type(None))
    o = OracleWRSN(scenario_of(g), num_agent=0)
    sg = o.static_graph()
    n = sc.N
    assert n == int(g["N"])
    assert np.array_equal(np.asarray(st["nbr_ptr"])[:n + 1], sg["nbr_ptr"]) and np.array_equal(st["nbr_idx"], sg["nbr_idx"])
    assert np.array_equal(np.asarray(st["tgt_ptr"])[:n + 1], sg["tgt_ptr"]) and np.array_equal(st["tgt_idx"], sg["tgt_idx"])
    assert np.array_equal(np.asarray(st["direct"])[:n].astype(np.int32), sg["direct"])
    assert sorted(np.nonzero(np.asarray(st["direct"])[:n])[0].tolist()) == sorted(int(x) for x in g["direct"])


@needs_reference
def test_all_nine_shipped_scenarios_load_and_match_the_oracle_graph():
    """L0: neighbour / target / base-station-direct sets of every shipped scenario (bacgiang_* through the fix-up switch)
    equal the oracle's, which restates Node.probe_neighbors / probe_targets / BaseStation.probe_neighbors."""
    from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict
    files = sorted(glob.glob(os.path.join(SHIPPED, "*.yaml")))
    assert len(files) == 9
    mc = load_mc_type(None)
    fixed = 0
    for f in files:
        raw = yaml.safe_load(open(f))
        if "max_time" not in raw:
            with pytest.raises(KeyError):
                Scenario.load_yaml(f)
            fixed += 1
        sc = Scenario.load_yaml(f, default_max_time=SHIPPED_MAX_TIME)
        st = build_static(sc, mc)
        o = OracleWRSN(scenario_from_dict(dict(raw, max_time=raw.get("max_time", SHIPPED_MAX_TIME))), num_agent=0)
        g = o.static_graph()
        n = sc.N
        assert np.array_equal(np.asarray(st["nbr_ptr"])[:n + 1], g["nbr_ptr"]) and np.array_equal(st["nbr_idx"], g["nbr_idx"]), f
        assert np.array_equal(np.asarray(st["tgt_ptr"])[:n + 1], g["tgt_ptr"]) and np.array_equal(st["tgt_idx"], g["tgt_idx"]), f
        assert np.array_equal(np.asarray(st["direct"])[:n].astype(np.int32), g["direct"]), f
    assert fixed == 4                                                  # bacgiang_50 / 100 / 150 / 200
