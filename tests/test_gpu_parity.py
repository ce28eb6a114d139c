"""Parity tests proper: the sm_100a kernels, called through the C ABI (libwrsn_b200.so), against the reference's
golden fixtures and the C oracle.  Run on the B200 box:  python -m pytest tests -m gpu"""
import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, _lib, synthetic
from tests import helpers, parity_cases as pc
from tests.helpers import golden_names

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module", autouse=True)
def cuda_library():
    L = helpers.use_cuda_build()        # raises if the extension is missing: no fallback
    assert not helpers.is_host_build(L)
    assert torch.cuda.is_available()
    yield


@pytest.mark.parametrize("name", golden_names("net_"))
def test_pure_network_golden(name):
    exact, total = pc.check_pure_network(name, DEV, replicas=2)
    assert exact == total


@pytest.mark.parametrize("name", golden_names("ep_"))
def test_episode_golden(name):
    pc.check_episode(name, DEV, check_obs=True)


def test_batched_replicas_identical():
    pc.check_episode("ep_edge_n50", DEV, replicas=5)


@pytest.mark.parametrize("seed", [0, 1])
def test_random_episodes_vs_oracle(seed):
    sc = synthetic(num_nodes=60, num_targets=70, seed=10 + seed)
    n_dec, cnt = pc.check_vs_oracle(sc, DEV, num_envs=8, steps=40, seed=seed, check_obs=(seed == 0))
    assert n_dec > 100


def test_heterogeneous_scenarios_vs_oracle():
    scs = [synthetic(num_nodes=48, num_targets=48, seed=s) for s in (21, 22, 23)]
    pc.check_vs_oracle(scs, DEV, num_envs=9, steps=25, seed=5)


def test_long_charging_and_deaths_vs_oracle():
    sc = synthetic(num_nodes=40, num_targets=120, seed=3, num_gateways=2)
    n_dec, cnt = pc.check_vs_oracle(sc, DEV, num_envs=6, steps=60, seed=9, scale2=0.5)
    assert cnt["serial_ticks"] >= 1


def test_small_charger_exhaustion_vs_oracle():
    mc = dict(capacity=2500, threshold=0, velocity=5, pm=1, charging_range=27, alpha=4500, beta=30, epsilon=1e-10)
    sc = synthetic(num_nodes=50, num_targets=50, seed=4)
    pc.check_vs_oracle(sc, DEV, num_envs=6, steps=50, seed=2, mc=mc, scale2=0.01)


def test_deaths_after_network_operate_stopped():
    """hanoi1000n50 far past the end of Network.operate: four more nodes die while the levels are stale."""
    from tests.helpers import golden
    sc = pc.sc_from_golden(golden("net_hanoi1000n50"))
    cnt, dead = pc.check_network_after_operate_stopped(sc, DEV, horizon=12000.0, every=100.0)
    assert dead >= 5 and cnt["stale_rebuilds"] >= 4


def test_rollout_step_equals_manual_loop():
    scs = [synthetic(num_nodes=40, num_targets=120, seed=s, num_gateways=2) for s in (3, 4)]
    resets = pc.check_rollout_step(scs, DEV, num_envs=16, steps=120, seed=1, with_obs=True)
    assert resets >= 3


@pytest.mark.parametrize("threads", [32, 128])
def test_batches_equal_event_path(threads):
    """Whole-cycle batches == the event-by-event path, byte for byte (node rows, clock, insertion counters)."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + s) for s in range(4)]
    a = pc.check_batches_equal_event_path(scs, DEV, num_envs=64, steps=300, seed=1, scale2=0.05, threads=threads)
    assert a["batched_ticks"] > 0.25 * a["ticks"]
    scs = [synthetic(num_nodes=40, num_targets=120, seed=s, num_gateways=2) for s in (3, 4)]
    b = pc.check_batches_equal_event_path(scs, DEV, num_envs=32, steps=150, seed=1, threads=threads)
    assert b["episode_ends"] >= 8


def test_batches_and_death_ticks_equal_event_path_300_nodes():
    """Several nodes per thread (300 nodes on 64 threads), long charges, episodes that end in deaths: batches and the
    piecewise death tick against the event-by-event path with the plain serial tick, byte for byte."""
    scs = [synthetic(num_nodes=300, num_targets=300, seed=40 + s, num_gateways=5) for s in range(2)]
    c = pc.check_batches_equal_event_path(scs, DEV, num_envs=24, steps=260, seed=3, num_agent=4, scale2=0.2, threads=64)
    assert c["split_death_ticks"] >= 1 or c["episode_ends"] >= 1


def test_pure_network_batches():
    from tests.helpers import golden
    sc = pc.sc_from_golden(golden("net_hanoi1000n50"))
    cnt = pc.check_pure_network_batches(sc, DEV, horizon=12500.0, every=37.0)
    assert cnt["batched_ticks"] > 0.6 * cnt["ticks"] and cnt["split_death_ticks"] >= 5


@pytest.mark.parametrize("threads", [32, 64, 128])
def test_group_size_independent(threads):
    """The result must not depend on how many threads share an environment."""
    sc = synthetic(num_nodes=100, num_targets=100, seed=7)
    rng = np.random.default_rng(3)
    acts = rng.uniform(0, 1, size=(30, 4, 3)); acts[..., 2] *= 0.05
    outs = []
    for th in (32, threads):
        env = BatchedWRSN(sc, num_agent=3, num_envs=4, device=DEV, threads=th)
        req = env.reset()
        rec = []
        for k in range(30):
            a = req.agent_id.clone()
            req = env.step(torch.where(a >= 0, a, torch.full_like(a, -1)), torch.as_tensor(acts[k], device=DEV), mask=(a >= 0))
            rec.append((req.agent_id.cpu().numpy().copy(), req.now.cpu().numpy().copy(), env.view("energy").cpu().numpy().copy()))
        outs.append(rec)
    for (a0, n0, e0), (a1, n1, e1) in zip(*outs):
        assert np.array_equal(a0, a1) and np.array_equal(n0, n1) and np.array_equal(e0, e1)


def test_full_size_properties():
    """BASELINE config 2 size (100 nodes / 3 chargers / 4096 environments): size-independent properties.
    Replicated environments fed identical actions must stay bit-identical; energies stay inside
    [threshold, capacity]; dead nodes never come back; time never runs backwards."""
    sc = synthetic(num_nodes=100, num_targets=100, seed=1)
    B = 4096
    env = BatchedWRSN(sc, num_agent=3, num_envs=B, device=DEV)
    rng = np.random.default_rng(0)
    req = env.reset()
    prev_now = req.now.clone()
    prev_status = env.view("status").clone()
    for k in range(12):
        a = rng.uniform(0, 1, size=(2, 3)); a[:, 2] *= 0.05
        act = torch.as_tensor(np.concatenate([np.tile(a[0], (B // 2, 1)), np.tile(a[1], (B // 2, 1))]), device=DEV)
        aid = req.agent_id.clone()
        req = env.step(aid, act, mask=(aid >= 0))
        e = env.view("energy")
        assert float(e.min()) >= 540.0 and float(e.max()) <= 10800.0
        assert bool((req.now >= prev_now).all())
        st = env.view("status")
        assert bool((st <= prev_status).all())
        prev_now, prev_status = req.now.clone(), st.clone()
        for half in (slice(0, B // 2), slice(B // 2, B)):
            assert bool((e[half] == e[half][0:1]).all())
            assert bool((req.agent_id[half] == req.agent_id[half][0]).all())
            assert bool((req.now[half] == req.now[half][0]).all())
    assert float(env.hdr("ERR").max()) == 0.0
    obs = env.get_state()
    assert obs.shape == (B, 4, 100, 100) and bool(torch.isfinite(obs).all())
    assert bool((obs[0] == obs[1]).all())


@pytest.mark.parametrize("nodes,targets,chargers,envs,steps", [(500, 500, 5, 3, 30), (1000, 1000, 10, 2, 45)])
def test_large_configs_vs_oracle(nodes, targets, chargers, envs, steps):
    """BASELINE configs 4 and 5 (500 nodes / 5 chargers, 1000 nodes / 10 chargers): the multi-warp build
    (128 / 256 threads per environment) against the oracle on a few environments and decisions."""
    sc = synthetic(num_nodes=nodes, num_targets=targets, seed=nodes, num_gateways=max(3, nodes // 40))
    n_dec, cnt = pc.check_vs_oracle(sc, DEV, num_envs=envs, steps=steps, seed=4, num_agent=chargers, check_obs=(nodes == 500))
    assert n_dec >= envs * 15


def test_charge_kernel_vs_reference_statements():
    """wrsn_k_charge: warp per environment, chargers staged in shared memory, per-charger sums in node order through ballot /
    shuffle — bit-exact with Node.charger_connection over MobileCharger.charge's connected nodes."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + s) for s in range(3)]
    assert pc.check_charge_kernel(scs, DEV, num_envs=9, steps=40, seed=2) > 50
    scs = [synthetic(num_nodes=300, num_targets=300, seed=40, num_gateways=5)]
    assert pc.check_charge_kernel(scs, DEV, num_envs=3, steps=20, seed=3, num_agent=5) > 10


# ------------------------------------------------------------------ round 2: the bench's own workload, budgets, shards, per-tick kernels
BENCH_SCENARIOS = [1000, 1001, 1002, 1003]           # bench.py: synthetic(100, 100, seed=1000 + k), 3 chargers


@pytest.mark.parametrize("threads", [32, 64])
def test_bench_scenarios_vs_oracle_uniform_actions(threads):
    """bench.py's exact scenarios (--actions uniform law), 64 environments x 60 steps against the oracle, float32 raster at
    1e-5 of the channel maximum — on one warp per environment (the bench's build) and on two."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS]
    n_dec, cnt = pc.check_vs_oracle(scs, DEV, num_envs=64, steps=60, seed=11, obs32=True, threads=threads)
    assert n_dec > 64 * 50


def test_bench_scenarios_vs_oracle_random_controller():
    """The headline workload as bench.py drives it: RandomController density map of the float32 observation, decoded on the
    device, 64 environments x 60 steps; the oracle is fed the decoded actions.  Agent ids, times, termination, status / level /
    coverage sets exact, energies 1e-9, reward 1e-9 (spec 1e-6): update_reward is active almost every second here."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS]
    n_dec, cnt = pc.check_vs_oracle(scs, DEV, num_envs=64, steps=60, seed=12, controller=True, obs32=True)
    assert n_dec > 64 * 40 and cnt["batched_ticks"] > 0.5 * cnt["ticks"]


@pytest.mark.parametrize("threads,budget,rounds", [(32, 25, 0), (64, 60, 0), (32, 160, 0), (32, 40, 1), (32, 100, 2), (64, 30, 3)])
def test_step_budget_only_cuts_steps_into_launches(threads, budget, rounds):
    """wrsn_dims.step_budget / step_rounds (events kernel + batch kernel): same requests, same records as the unbudgeted run."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS]
    n = pc.check_budget_equals_unbudgeted(scs, DEV, num_envs=32, calls=80, seed=5, budget=budget, scale2=0.1, threads=threads,
                                          rounds=rounds)
    assert n > 10
    scs = [synthetic(num_nodes=40, num_targets=120, seed=s, num_gateways=2) for s in (3, 4)]
    pc.check_budget_equals_unbudgeted(scs, DEV, num_envs=8, calls=60, seed=6, budget=budget, scale2=0.3, threads=threads, rounds=rounds)


def test_sharded_equals_unsharded_records():
    """Two / three simulators holding contiguous blocks of the environments == one simulator holding all of them, byte for
    byte (SURVEY 8e: environments shard by index, nothing is exchanged) — also with a step budget."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS[:3]]
    pc.check_sharded_equals_unsharded(scs, DEV, num_envs=50, steps=60, seed=2, world=2)
    pc.check_sharded_equals_unsharded(scs, DEV, num_envs=50, steps=60, seed=3, world=3, budget=40)
    pc.check_sharded_equals_unsharded(scs, DEV, num_envs=50, steps=60, seed=4, world=2, budget=60, rounds=2)


@pytest.mark.parametrize("name,t_from,t_to", [("net_hanoi1000n200", 512, 524), ("net_hanoi1000n100", 1598, 1608)])
def test_tick_kernels_across_a_death_tick(name, t_from, t_to):
    """Ladder L1 / L2: wrsn_k_drain / wrsn_k_bookkeep / wrsn_k_bfs launched by hand, tick by tick, across the death ticks of the
    shipped scenarios (SURVEY 8c table: hanoi1000n200 518.5, hanoi1000n100 1602.5), against the oracle."""
    assert pc.check_tick_kernels(name, DEV, t_from, t_to) >= 1


def test_reward_kernel_vs_reference_statements():
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS[:2]]
    assert pc.check_reward_kernel(scs, DEV, num_envs=8, steps=30, seed=3) > 20


@pytest.mark.parametrize("chunk", range(5))
def test_fuzz_engine_vs_oracle(chunk):
    """Ladder L7 on the device: 10 random configurations per case (20-90 nodes, 10-150 targets, 1-4 chargers, charge fractions
    up to 1, 30-160 steps, every fourth with observations) against the C restatement, decision by decision."""
    n = 0
    for seed in range(5000 + 10 * chunk, 5010 + 10 * chunk):
        rng = np.random.default_rng(seed)
        N, T, M = int(rng.integers(20, 90)), int(rng.integers(10, 150)), int(rng.integers(1, 5))
        gw, scale2 = int(rng.integers(2, 5)), float(rng.choice([0.02, 0.1, 0.5, 1.0]))
        steps = int(rng.integers(30, 160))
        sc = synthetic(num_nodes=N, num_targets=T, seed=seed, num_gateways=gw)
        n_dec, _ = pc.check_vs_oracle(sc, DEV, num_envs=3, steps=steps, seed=seed, num_agent=M, scale2=scale2,
                                      check_obs=seed % 4 == 0)
        n += n_dec
    assert n > 300


def test_simulator_on_a_device_that_is_not_current():
    """The launches must follow the simulator's device, not the CUDA runtime's current one (needs two GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    sc = synthetic(num_nodes=60, num_targets=60, seed=3)
    rng = np.random.default_rng(0)
    acts = rng.uniform(0, 1, size=(10, 4, 3)); acts[..., 2] *= 0.05
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        with torch.cuda.device(0):                   # cuda:0 stays current
            env = BatchedWRSN(sc, num_agent=3, num_envs=4, device=dev)
            env.reset()
            for k in range(10):
                env.rollout_step(torch.as_tensor(acts[k], device=dev))
            obs = env.get_state()
            outs.append((env.state.cpu(), obs.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_launch_order_changes_no_result():
    """k_step_order (launches of >= 2048 rows are taken longest predicted step first): 2304 environments — 768 replicas of three
    scenarios, every replica of a scenario fed the same actions — against 3 environments stepped in index order (no ordering below
    2048 rows): every replica's requests and record equal, byte for byte, those of its scenario's single environment."""
    scs = [synthetic(num_nodes=100, num_targets=100, seed=s) for s in BENCH_SCENARIOS[:3]]
    R, steps = 768, 40
    big = BatchedWRSN(scs, num_agent=3, num_envs=3 * R, device=DEV, scenario_index=np.arange(3 * R) % 3, step_budget=60)
    small = BatchedWRSN(scs, num_agent=3, num_envs=3, device=DEV, step_budget=60)
    rng = np.random.default_rng(11)
    acts = rng.uniform(0.0, 1.0, size=(steps, 3, 3)); acts[..., 2] *= 0.1
    end = int(big._foff[big.E["WRSN_F_SCRATCH"]])
    big.reset(); small.reset()
    for k in range(steps):
        small.rollout_step(torch.as_tensor(acts[k], device=DEV))
        big.rollout_step(torch.as_tensor(np.tile(acts[k], (R, 1)), device=DEV))
        for f in ("agent_id", "terminal", "now", "reward", "flags"):
            x, y = getattr(big.req, f).view(R, 3), getattr(small.req, f).view(1, 3)
            assert bool(((x == y) | ((x != x) & (y != y))).all()), (k, f)
        assert torch.equal(big.state[:, :end].view(R, 3, end), small.state[:, :end].view(1, 3, end).expand(R, 3, end)), k
    assert int((big.req.order.sort().values != torch.arange(3 * R, device=DEV, dtype=torch.int32)).sum()) == 0   # a permutation
