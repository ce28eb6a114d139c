"""Crowded fields: many chargers, wide charging ranges, mass deaths and full node slots.

The step kernel has fixed-size paths with a fallback for when they fill up: the incentive sums by pair list (at most
WRSN_PAIR_MAX = 32 (charging charger, connected alive node) pairs, else one thread per charger), the irregular-node table of a
whole-cycle batch (WRSN_SPEC_MAX = 16 entries, else the second runs event by event), the piecewise death tick (at most 4
endangered nodes, else the serial tick), 16 chargers per environment, and 4 node slots per lane on one warp or 9 per thread on
several.  Every case here drives one of them past its limit and compares with the C oracle (ids, times, sets and termination
exact, energies 1e-9, reward 1e-9) or, byte for byte, with another path of the same library.

The host build runs every environment on one lane, so its incentive sums always take the one-thread fallback; the one-lane-per-pair
and one-lane-per-charger sums run on the GPU only (``-m gpu``).  Each test also counts, from the record at every request, how often
it reached the regime it is about (the witnesses below) and fails if that count is too small: a change to ``synthetic()`` or to a
default must not turn it into a test of something else."""
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, Scenario, synthetic
from multi_agent_rl_wrsn_b200.scenario import DEFAULT_MC, DEFAULT_NODE_PHY
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
PAIR_MAX, SPEC_MAX = 32, 16                          # WRSN_PAIR_MAX, WRSN_SPEC_MAX (wrsn_layout.h)
BENCH_SEEDS = (1000, 1001, 1002, 1003)               # bench.py's scenarios: synthetic(100, 100, seed=1000 + k)


@pytest.fixture(scope="module")
def emu_built():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)


@pytest.fixture
def dev(request, emu_built):
    """The host emulation for "cpu", the CUDA library (no fallback) for the GPU."""
    if request.param == "cpu":
        helpers.use_host_build()
        yield "cpu"
        helpers.use_cuda_build_lazy()
    else:
        L = helpers.use_cuda_build()
        assert not helpers.is_host_build(L) and torch.cuda.is_available()
        yield request.param


def cpu(*args, **kw):
    return pytest.param("cpu", *args, **kw)


def gpu(*args, **kw):
    return pytest.param(GPU, *args, marks=pytest.mark.gpu, **kw)


def mc_of(charging_range):
    return dict(DEFAULT_MC, charging_range=float(charging_range))


_SCEN = {}


def scenario(N, seed, gateways=3):
    """synthetic() once per module and arguments (1152 nodes take seconds to place)."""
    key = (N, seed, gateways)
    if key not in _SCEN:
        _SCEN[key] = synthetic(num_nodes=N, num_targets=N, seed=seed, num_gateways=gateways)
    return _SCEN[key]


def bench_scenarios():
    return [scenario(100, s) for s in BENCH_SEEDS]


# ------------------------------------------------------------------ witnesses, read from the record at every request
def pairs(env):
    """Per row: the (charger a, node i) with mc STATUS != 0 and TYPE != 0, bit i set in conn_words[a] and status[i] == 1 — the
    predicate of reward_pair_list, i.e. the length of the incentive sums' pair list."""
    cw = env.view("conn_words")[:, :env.M].to(torch.int64) & 0xFFFFFFFF
    bits = ((cw.unsqueeze(-1) >> torch.arange(32, device=env.device)) & 1).reshape(env.B, env.M, -1)[:, :, :env.N] != 0
    on = (env.mc("STATUS") != 0) & (env.mc("TYPE") != 0)
    alive = env.view("status") == 1
    return (bits & on.unsqueeze(-1) & alive.unsqueeze(1)).sum((1, 2)).cpu().numpy()


def charged(env):
    """Per row: alive nodes with energyRR != 0 (a lower bound on the irregular-node table of a batch)."""
    return ((env.view("status") == 1) & (env.view("rr") != 0)).sum(1).cpu().numpy()


class Witness:
    """Counts requests by regime; pass it as the checkers' ``probe``."""

    def __init__(self):
        self.pairs, self.charged, self.threads = [], [], set()

    def __call__(self, env, rows=None):
        p, c = pairs(env), charged(env)
        if rows is not None:
            p, c = p[rows], c[rows]
        self.pairs += p.tolist()
        self.charged += c.tolist()
        self.threads.add(env.dims.threads)

    def listed(self, lo=4):
        """requests whose incentive sums take the pair list on the GPU with at least `lo` lanes"""
        return sum(lo <= p <= PAIR_MAX for p in self.pairs)

    def fallback(self):
        """requests whose incentive sums take the one-thread-per-charger fallback"""
        return sum(p > PAIR_MAX for p in self.pairs)

    def table_full(self):
        """requests with more charged nodes than the irregular-node table of a batch holds"""
        return sum(c > SPEC_MAX for c in self.charged)

    def __repr__(self):
        return "requests %d, listed (4-32 pairs) %d, fallback (> 32) %d, max pairs %d, table full %d, max charged %d" % (
            len(self.pairs), self.listed(), self.fallback(), max(self.pairs, default=0), self.table_full(),
            max(self.charged, default=0))


# ------------------------------------------------------------------ 1. the pair list and its fallback, swept against the oracle
SWEEP_M, SWEEP_R, SWEEP_S2 = (4, 8, 16), (27, 60, 120, 250), (0.05, 0.1, 0.2, 0.3)
SWEEP_CASES = ([gpu(M, R, th, 16, 60, id="gpu-M%d-R%d-t%d" % (M, R, th)) for M in SWEEP_M for R in SWEEP_R for th in (32, 64)]
               + [gpu(16, 120, 128, 16, 60, id="gpu-M16-R120-t128")]
               + [cpu(M, R, 0, 4, 40, id="cpu-M%d-R%d" % (M, R)) for M, R in ((16, 27), (8, 60), (16, 120), (4, 250))])


@pytest.mark.parametrize("dev,M,R,threads,rows,steps", SWEEP_CASES, indirect=["dev"])
def test_pair_list_sweep_vs_oracle(dev, M, R, threads, rows, steps):
    """The bench's 100-node scenarios under uniform actions with 4 / 8 / 16 chargers whose charging range grows from the default
    27 m to 250 m: from a few (charging charger, connected alive node) pairs per tick — one lane per pair on the GPU — to hundreds,
    beyond WRSN_PAIR_MAX, where one thread per charger sums its nodes."""
    i, j = SWEEP_M.index(M), SWEEP_R.index(R)
    w = Witness()
    n_dec, _ = pc.check_vs_oracle(bench_scenarios(), dev, num_envs=rows, steps=steps, seed=100 + 4 * i + j, num_agent=M,
                                  mc=mc_of(R), scale2=SWEEP_S2[(i + j) % 4], threads=threads, probe=w)
    n = len(w.pairs)
    assert n_dec >= rows * steps // 3 and (not threads or w.threads == {threads}), (n_dec, w.threads)
    if R <= 27:
        assert w.listed(lo=2) >= 0.2 * n and w.fallback() == 0, w           # several lanes of the list
    elif R <= 60:
        assert w.listed(lo=14) >= 0.02 * n, w                               # most of a warp's lanes (27 m never gets there)
    else:
        assert w.fallback() >= 0.3 * n, w                                   # past WRSN_PAIR_MAX


# ------------------------------------------------------------------ 2. whole-cycle batches with a full irregular-node table
BATCH_CASES = ([gpu(R, th, 32, 100, id="gpu-R%d-t%d" % (R, th)) for R in (120, 250) for th in (32, 64)]
               + [cpu(120, 0, 4, 60, id="cpu-R120")])


@pytest.mark.parametrize("dev,R,threads,rows,steps", BATCH_CASES, indirect=["dev"])
def test_batches_equal_event_path_crowded(dev, R, threads, rows, steps):
    """16 chargers charging dozens of nodes at once: a batch's irregular-node table (WRSN_SPEC_MAX entries) overflows and that
    second runs event by event, while the batches around it go on.  Every byte of the record must equal the event path's."""
    w = Witness()
    cnt = pc.check_batches_equal_event_path(bench_scenarios(), dev, num_envs=rows, steps=steps, seed=21, num_agent=16, scale2=0.1,
                                            threads=threads, mc=mc_of(R), probe=w)
    assert w.table_full() >= 0.2 * len(w.charged) and w.fallback() >= 0.2 * len(w.pairs), w
    assert cnt["batched_ticks"] > 0, cnt


# ------------------------------------------------------------------ 3. step budgets and split rounds on the same field
BUDGET_CASES = ([gpu(b, r, 32, 60, id="gpu-b%d-r%d" % (b, r)) for b in (25, 60) for r in (0, 2)]
                + [cpu(25, 2, 4, 40, id="cpu-b25-r2"), cpu(60, 0, 4, 40, id="cpu-b60-r0")])


@pytest.mark.parametrize("dev,budget,rounds,rows,calls", BUDGET_CASES, indirect=["dev"])
def test_budget_equals_unbudgeted_crowded(dev, budget, rounds, rows, calls):
    """A step cut into launches by a budget (and split between the events and the batch kernel) resumes exactly, also inside the
    seconds a full table sends back to the event path: every request and every byte of the record as without a budget."""
    w = Witness()
    n = pc.check_budget_equals_unbudgeted(bench_scenarios(), dev, num_envs=rows, calls=calls, seed=22, budget=budget, num_agent=16,
                                          scale2=0.1, rounds=rounds, mc=mc_of(120), probe=w)
    assert n >= 2 * rows, n
    assert w.table_full() >= 0.2 * len(w.charged) and w.fallback() >= 0.2 * len(w.pairs), w


# ------------------------------------------------------------------ 4. simultaneous deaths
BS = np.array([500.0, 500.0])
ORBIT4 = [(50, 0), (0, 50), (-50, 0), (0, -50)]
ORBIT8 = [(30, 40), (-40, -30), (40, -30), (-30, 40), (40, 30), (-30, -40), (30, -40), (-40, 30)]


def orbit(kind):
    """Nodes on orbits of the square's symmetry group, all exactly 50 m from the base station, each with its target 1.2 times as
    far out along its ray: every node of an orbit spends the same energy in the same order, so they all die in the same tick."""
    off = np.array({"o4": ORBIT4, "o8": ORBIT8, "o4+o8": ORBIT4 + ORBIT8}[kind], np.float64)
    return Scenario(nodes=BS + off, targets=BS + 1.2 * off, base_station=BS.copy(), node_phy_spe=dict(DEFAULT_NODE_PHY), seed=0,
                    max_time=604800.0, name=kind)


DEATH_CASES = [cpu(k, 0, id="cpu-" + k) for k in ("o4", "o8", "o4+o8")] + \
              [gpu(k, th, id="gpu-%s-t%d" % (k, th)) for k in ("o4", "o8", "o4+o8") for th in (32, 64)]


@pytest.mark.parametrize("dev,kind,threads", DEATH_CASES, indirect=["dev"])
def test_simultaneous_deaths_vs_oracle(dev, kind, threads):
    """4 nodes die in one tick: the piecewise death tick (at most 4 endangered nodes).  8 and 12: the serial tick."""
    sc = orbit(kind)
    cnt, dead = pc.check_network_after_operate_stopped(sc, dev, horizon=400000.0, every=997.0, threads=threads)
    assert dead == sc.N, dead
    if kind == "o4":
        assert cnt["split_death_ticks"] >= 1, cnt
    else:
        assert cnt["serial_ticks"] >= 1 and cnt["split_death_ticks"] == 0, cnt


@pytest.mark.parametrize("dev,threads", [cpu(0, id="cpu"), gpu(32, id="gpu-t32"), gpu(64, id="gpu-t64")], indirect=["dev"])
def test_episode_ending_in_a_mass_death_vs_oracle(dev, threads):
    """An episode under uniform actions whose chargers reach no node (1 m charging range): the network runs down on its own and
    the episode ends at the request after all 8 nodes of the orbit died in the same tick."""
    alive = [[] for _ in range(2)]

    def probe(env, rows):
        st = (env.view("status") == 1).sum(1).tolist()
        for b in range(2):
            if rows[b]:
                alive[b].append((st[b], int(env.req.terminal[b])))
    n_dec, cnt = pc.check_vs_oracle(orbit("o8"), dev, num_envs=2, steps=400, seed=1, num_agent=2, mc=mc_of(1.0), scale2=1.0,
                                    threads=threads, probe=probe)
    for b in range(2):
        assert alive[b][-1] == (0, 1) and alive[b][-2][0] == 8, alive[b][-3:]
    assert cnt["serial_ticks"] >= 2 and n_dec >= 300, (cnt, n_dec)


# ------------------------------------------------------------------ 5. 16 chargers on multi-warp rows
WIDE_CASES = [gpu(N, th, 3, id="gpu-N%d-t%d" % (N, th)) for N in (300, 500) for th in (64, 128)] + [cpu(300, 0, 2, id="cpu-N300")]


@pytest.mark.parametrize("dev,N,threads,rows", WIDE_CASES, indirect=["dev"])
def test_sixteen_chargers_multi_warp_vs_oracle(dev, N, threads, rows):
    sc = scenario(N, seed=N, gateways=max(3, N // 40))
    w = Witness()
    n_dec, _ = pc.check_vs_oracle(sc, dev, num_envs=rows, steps=30, seed=N + 1, num_agent=16, mc=mc_of(120), scale2=0.1,
                                  threads=threads, probe=w)
    assert n_dec >= rows * 20 and w.fallback() >= 0.3 * len(w.pairs), (n_dec, w)
    assert w.threads == {threads} if threads else min(w.threads) > 32, w.threads


# ------------------------------------------------------------------ 6. node slots at their limits
SLOT_CASES = ([cpu(128, 32, 32, id="cpu-N128-t32"), cpu(129, 0, 64, id="cpu-N129-default")]
              + [gpu(N, th, want, id="gpu-N%d-%s" % (N, "t%d" % th if th else "default"))
                 for N, th, want in ((128, 32, 32), (576, 64, 64), (1152, 128, 128), (129, 0, 64), (1153, 0, 256))])


def slot_scenario(N):
    return scenario(N, seed=N, gateways=max(3, N // 40))


@pytest.mark.parametrize("dev,N,threads,want", SLOT_CASES, indirect=["dev"])
def test_node_slots_at_their_limits_vs_oracle(dev, N, threads, want):
    """Every node slot of a row in use: 4 per lane on one warp (128 nodes), 9 per thread on 64 / 128 threads (576 / 1152), and one
    node more than a size's slots, where the default thread count must step up (129 -> 64 threads, 1153 -> 256)."""
    w = Witness()
    n_dec, _ = pc.check_vs_oracle(slot_scenario(N), dev, num_envs=2, steps=25, seed=9, num_agent=3, scale2=0.05, threads=threads,
                                  probe=w)
    assert w.threads == {want}, w.threads
    if threads:
        assert N == want * (4 if want == 32 else 9)                     # every slot in use
    else:
        assert N == (want // 2) * (4 if want == 64 else 9) + 1          # one node more than half as many threads hold
    assert n_dec >= 10, n_dec


@pytest.mark.gpu
@pytest.mark.parametrize("dev,N,group", [(GPU, 128, (32, 64, 128)), (GPU, 576, (64, 128, 256))], indirect=["dev"])
def test_node_slots_group_size_independent(dev, N, group):
    """The same rows on different thread counts, one of them with every slot in use: every request and every byte of the record
    must be the same, apart from update_reward's outputs (the reward and the chargers' exclusive reward), which agree to 1e-9:
    the softmax's sums over the nodes are taken per thread and then across threads, so their rounding follows the thread count."""
    rng = np.random.default_rng(N)
    acts = rng.uniform(0.0, 1.0, size=(30, 2, 3))
    acts[..., 2] *= 0.05
    envs = [BatchedWRSN(slot_scenario(N), num_agent=3, num_envs=2, device=dev, threads=th) for th in group]
    assert sorted(e.dims.threads for e in envs) == sorted(group)
    excl = envs[0].E["WRSN_MC_EXCL"]

    def record(e):
        mc = e.view("mc").cpu().numpy().copy()
        out = {f: e.view(f).cpu().numpy().copy() for f in pc._STATE_FIELDS if f != "mc"}
        out["excl"], out["reward"] = mc[:, :, excl].copy(), e.req.reward.cpu().numpy().copy()
        mc[:, :, excl] = 0.0
        out["mc"] = mc
        out.update({f: getattr(e.req, f).cpu().numpy().copy() for f in ("agent_id", "terminal", "now", "action", "flags")})
        return out
    for e in envs:
        e.reset()
    for k in range(30):
        for e in envs:
            e.rollout_step(torch.as_tensor(acts[k], device=dev))
        want = record(envs[0])
        for e in envs[1:]:
            got = record(e)
            for f, v in want.items():
                if f in ("excl", "reward"):
                    atol = 1e-12 * max(1.0, float(np.abs(want["excl"]).max()))
                    np.testing.assert_allclose(got[f], v, rtol=1e-9, atol=atol, err_msg=str((k, e.dims.threads, f)))
                else:
                    assert np.array_equal(got[f].view(np.uint8), v.view(np.uint8)), (k, e.dims.threads, f)
    assert all(float(e.hdr("ERR").max()) == 0.0 for e in envs)


# ------------------------------------------------------------------ 7. the charging model on dense connections
class Cover:
    """Per check and charger: the alive nodes within its charging range, and how many distinct places the chargers are at."""

    def __init__(self):
        self.counts, self.places = [], []

    def __call__(self, env):
        sid, status = env.scen_id.cpu().numpy(), env.view("status").cpu().numpy()
        mx, my, R = env.mc("X").cpu().numpy(), env.mc("Y").cpu().numpy(), env.mc_type["charging_range"]
        for b in range(env.B):
            xy = np.asarray(env.scenarios[sid[b]].nodes, np.float64)
            d = np.hypot(xy[None, :, 0] - mx[b][:, None], xy[None, :, 1] - my[b][:, None])
            self.counts.append(((d <= R) & (status[b][None] == 1)).sum(1))
            self.places.append(len(set(zip(mx[b].tolist(), my[b].tolist()))))


@pytest.mark.parametrize("dev,rows,steps", [cpu(2, 40, id="cpu"), gpu(9, 60, id="gpu")], indirect=["dev"])
def test_charge_kernel_dense_connections(dev, rows, steps):
    """wrsn_k_charge with 16 chargers of 250 m range spread over the field: each charger's sum runs over dozens of nodes (several
    ballot / shuffle rounds in node order on the GPU) and must equal the reference's statements to the last bits."""
    cover = Cover()
    pc.check_charge_kernel(bench_scenarios()[:3], dev, num_envs=rows, steps=steps, seed=4, num_agent=16, mc=mc_of(250), probe=cover)
    counts = np.array(cover.counts)
    spread = np.array(cover.places) >= 8
    assert spread.sum() >= 0.3 * len(spread) and (counts[spread] > 32).sum() >= 0.2 * counts[spread].size, (cover.places, counts)


# ------------------------------------------------------------------ 8. dense fuzz
def fuzz_case(seed):
    rng = np.random.default_rng(seed)
    N, M = int(rng.integers(20, 301)), int(rng.integers(1, 17))
    R, scale2 = float(rng.uniform(27.0, 300.0)), float(rng.choice([0.01, 0.1, 0.5, 1.0]))
    steps, gateways = int(rng.integers(30, 121)), int(rng.integers(2, 5)) + N // 100
    return scenario(N, seed=seed, gateways=gateways), M, R, scale2, steps


FUZZ_CASES = [cpu(range(7100, 7104), id="cpu")] + [gpu(range(7000 + 10 * c, 7010 + 10 * c), id="gpu-%d" % c) for c in range(3)]


@pytest.mark.parametrize("dev,seeds", FUZZ_CASES, indirect=["dev"])
def test_dense_fuzz_vs_oracle(dev, seeds):
    """Random crowded configurations — 20-300 nodes, 1-16 chargers of 27-300 m range, charge fractions up to 1 — against the
    oracle, every fourth also with observations."""
    w = Witness()
    n = 0
    for seed in seeds:
        sc, M, R, scale2, steps = fuzz_case(seed)
        n_dec, _ = pc.check_vs_oracle(sc, dev, num_envs=3, steps=steps, seed=seed, num_agent=M, mc=mc_of(R), scale2=scale2,
                                      check_obs=seed % 4 == 0, probe=w)
        n += n_dec
    assert n >= 40 * len(seeds), n
    assert w.listed() >= 0.05 * len(w.pairs) and w.fallback() >= 0.1 * len(w.pairs), w
