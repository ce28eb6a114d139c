"""TEST INFRASTRUCTURE (not collected by pytest; needs a checkout of the reference: set WRSN_REFERENCE_ROOT): the C restatement of the
reference (oracle/wrsn_oracle.c) against the UNMODIFIED Python reference run under the oracle shims, on RANDOM synthetic
scenarios and action streams — beyond the 16 committed fixtures.  Decision by decision: agent id, terminal flag, env.now and
every node's status identical; reward, node energies, charger energies at 1e-9 relative.

    python tests/fuzz_oracle_vs_reference.py [--first-seed 0] [--count 6] [--decisions 10]

End of round 1: seeds 0-3 (8 decisions each) and 10-49 (15 each): 618 decisions, no difference."""
import argparse
import os
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from multi_agent_rl_wrsn_b200 import synthetic  # noqa: E402
from oracle import ref_runner  # noqa: E402
from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict  # noqa: E402


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--first-seed", type=int, default=0)
    p.add_argument("--count", type=int, default=6)
    p.add_argument("--decisions", type=int, default=10)
    a = p.parse_args()
    R = ref_runner.load_reference()
    cwd = os.getcwd()
    os.chdir(R.root)                                                      # the reference opens files relative to its root (SURVEY Q11)
    fails = n = 0
    t0 = time.time()
    try:
        for seed in range(a.first_seed, a.first_seed + a.count):
            rng = np.random.default_rng(seed)
            N, T, M = int(rng.integers(20, 45)), int(rng.integers(10, 60)), int(rng.integers(1, 4))
            scale2 = float(rng.choice([0.02, 0.1, 0.4]))
            sc = synthetic(num_nodes=N, num_targets=T, seed=500 + seed, num_gateways=int(rng.integers(2, 4)))
            with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
                path = f.name
            sc.save_yaml(path)
            try:
                ref = R.WRSN(scenario_path=path, agent_type_path=R.mc_type, num_agent=M, map_size=100, density_map=False)
                orc = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=M)
                rq, oq = ref.reset(), orc.reset(want_state=False)
                for k in range(a.decisions):
                    tag = (seed, k)
                    assert (rq["agent_id"] if rq["agent_id"] is not None else -1) == (oq["agent_id"] if oq["agent_id"] is not None else -1), tag
                    assert bool(rq["terminal"]) == oq["terminal"], tag
                    assert float(ref.env.now) == oq["now"], tag
                    nodes = orc.nodes()
                    e_ref = np.array([nd.energy for nd in ref.net.listNodes])
                    assert np.array_equal(np.array([nd.status for nd in ref.net.listNodes], np.uint8), nodes["status"]), tag
                    np.testing.assert_allclose(nodes["energy"], e_ref, rtol=1e-9, err_msg=str(tag))
                    np.testing.assert_allclose(orc.mcs()["energy"], [m.energy for m in ref.agents], rtol=1e-9, err_msg=str(tag))
                    if rq["agent_id"] is None:
                        break
                    if k > 0:
                        np.testing.assert_allclose(oq["reward"], rq["reward"], rtol=1e-9, atol=1e-15, err_msg=str(tag))
                    n += 1
                    act = rng.uniform(0, 1, 3)
                    act[2] *= scale2
                    rq, oq = ref.step(rq["agent_id"], act), orc.step(oq["agent_id"], act, want_state=False)
            except AssertionError as e:
                fails += 1
                print("FAIL", (seed, N, T, M, scale2), str(e)[:300], flush=True)
            finally:
                os.unlink(path)
            print("seed %d: N=%d T=%d M=%d ok so far %d decisions, %.0f s" % (seed, N, T, M, n, time.time() - t0), flush=True)
    finally:
        os.chdir(cwd)
    print("%d decisions compared, %d failing configurations" % (n, fails))
    return 1 if fails else 0


if __name__ == "__main__":
    sys.exit(main())
