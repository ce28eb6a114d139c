"""Host-side pieces of bench.py that run without a GPU: the workloads it builds and the reference arm's CPU sample."""
import argparse
import importlib.util
import os
import subprocess

import pytest

from tests.helpers import REPO


def _bench():
    spec = importlib.util.spec_from_file_location("_bench_mod", os.path.join(REPO, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _args(**kw):
    base = dict(nodes=100, targets=None, chargers=3, envs=4096, topologies=3, scenario=None, actions="controller")
    base.update(kw)
    return argparse.Namespace(**base)


def test_workloads():
    b = _bench()
    scs = b.scenarios_for(_args(), rank=1)
    assert len(scs) == 3 and all(s.N == 100 and s.T == 100 for s in scs)
    other = b.scenarios_for(_args(), rank=0)
    assert any((x.nodes != y.nodes).any() for x, y in zip(scs, other))          # every rank has its own topologies
    shipped = b.scenarios_for(_args(scenario="net_hanoi1000n100"), rank=0)      # the reference's hanoi1000n100.yaml (SURVEY 8c table)
    assert len(shipped) == 1 and (shipped[0].N, shipped[0].T) == (98, 100)
    assert "hanoi1000n100" in b.workload_name(_args(scenario="net_hanoi1000n100"))
    assert "100-node/3-charger" in b.workload_name(_args())


def test_cpu_sample_of_the_reference_arm():
    """One short single-core sample of the C restatement, as `cpu_baseline` / `--impl reference` take it."""
    b = _bench()
    out = b.cpu_baseline(_args(topologies=1, actions="uniform"), cores=1, budget_s=1.0)
    assert out["kind"] == "port" and out["cores"] == 1 and out["unit"] == b.UNIT and out["value"] > 10.0
    # the headline law: the RandomController map decoded by the reference's own numpy / scipy statements (slow: L-BFGS-B)
    out = b.cpu_baseline(_args(topologies=1), cores=1, budget_s=2.0)
    assert out["value"] > 0.5 and "RandomController" in out["sample"]
    assert "RandomController" in b.workload_name(_args()) and "uniform" in b.workload_name(_args(actions="uniform"))


def test_arguments():
    b = _bench()
    a = b.parse(["--steps", "7", "--warmup", "2", "--dump-outputs", "out"])
    assert (a.steps, a.warmup, a.dump_outputs) == (7, 2, "out")
    a = b.parse(["--workload", "ippo", "--steps", "2"])                      # IPPO: one timed step = one training iteration
    assert (a.steps, a.iterations) == (2, 2)
    assert (b.parse(["--workload", "ippo"]).steps, b.parse([]).steps) == (3, 60)
    for bad in (["--steps", "0"], ["--workload", "ippo", "--steps", "0"], ["--workload", "ippo", "--dump-outputs", "out"], ["--impl", "reference", "--dump-outputs", "out"]):
        with pytest.raises(SystemExit):
            b.parse(bad)


def test_dump_outputs(tmp_path):
    """--dump-outputs on two groups of environments stepped through the host emulation of the kernel source (tests/emu).  A small
    step budget of one work unit keeps the second group's steps in flight: rows without a request, whose reward, detail and action
    are NaN in the record, are written as 0.  A second dump with a smaller environment cap keeps a seeded sample of the rows."""
    import numpy as np
    import torch
    from multi_agent_rl_wrsn_b200 import BatchedWRSN, synthetic
    from tests import helpers
    subprocess.check_call(["make", "-C", os.path.join(REPO, "tests", "emu"), "libwrsn_emu.so"], stdout=subprocess.DEVNULL)
    helpers.use_host_build()
    try:
        b = _bench()
        S, Bg, G = 20, 40, 2
        scs = [synthetic(num_nodes=30, num_targets=30, seed=s) for s in (1, 2)]
        groups = [BatchedWRSN(scs, num_agent=2, num_envs=Bg, device="cpu", map_size=S, scenario_index=np.arange(Bg) % 2,
                              step_budget=budget) for budget in (0, 1)]
        obs = [torch.zeros((Bg, 4, S, S)) for _ in range(G)]
        act = [torch.zeros((Bg, 3), dtype=torch.float64) for _ in range(G)]
        g = torch.Generator().manual_seed(0)
        for env, o in zip(groups, obs):
            env.reset()
            env.get_state(out=o)
        for _ in range(5):
            for env, o, x in zip(groups, obs, act):
                torch.mul(torch.rand((Bg, 3), generator=g, dtype=torch.float64), torch.tensor([1.0, 1.0, 0.05]), out=x)
                env.rollout_step(x, o)
        b.dump_outputs(str(tmp_path / "all"), groups, act, obs)
        b.DUMP_MAX_ENVS = 50
        b.dump_outputs(str(tmp_path / "sampled"), groups, act, obs)
    finally:
        helpers.use_cuda_build_lazy()
    names = ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats")
    req = {name: torch.cat([getattr(env.req, name) for env in groups]).to(torch.float64).numpy() for name in names}
    has = req["agent_id"] >= 0
    assert has.any() and (~has).any()
    assert all(np.isnan(req[name][~has]).all() for name in ("reward", "detail", "action"))
    got = {p.name[:-4]: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(got) == {"request_" + name for name in names} | {"action", "env_rows", "observation", "observation_rows"}
    assert all(v.dtype in (np.float32, np.float64) and np.isfinite(v).all() for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    assert np.array_equal(got["env_rows"], np.arange(G * Bg))
    for name in names:
        assert np.array_equal(got["request_" + name][has], req[name][has]), name
        none = np.zeros_like(req[name][~has]) if name in ("reward", "detail", "action") else req[name][~has]
        assert np.array_equal(got["request_" + name][~has], none), name
    assert np.array_equal(got["action"], torch.cat(act).numpy())
    sampled = {p.name[:-4]: np.load(p) for p in (tmp_path / "sampled").iterdir()}
    env_rows = sampled["env_rows"].astype(np.int64)
    assert len(env_rows) == 50 and np.all(np.diff(env_rows) > 0) and env_rows.max() < G * Bg
    assert np.array_equal(sampled["request_now"], req["now"][env_rows]) and np.array_equal(sampled["action"], got["action"][env_rows])
    assert np.array_equal(sampled["observation_rows"], got["observation_rows"])
    rows = got["observation_rows"].astype(np.int64)
    assert len(rows) == b.DUMP_OBS_ROWS and np.all(np.diff(rows) > 0) and rows.min() >= 0 and rows.max() < G * Bg
    assert got["observation"].dtype == np.float32 and np.array_equal(got["observation"], torch.cat(obs).numpy()[rows])
    assert got["observation"].any()
