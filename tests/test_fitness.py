"""WRSN.get_network_fitness (``wrsn_fitness``, the step kernel's ``do_fitness``) against a restatement by another algorithm.

``do_fitness`` seeds every alive node with the bottleneck of its own routing path (the parent walk) and relaxes a widest-path
(max-min) fixpoint by pulling from its neighbours until no thread changes anything; the per-target values are an atomic max.
The C oracle runs a label-correcting search from the direct nodes, and ``oracle/fitness_oracle.py`` a label-setting one over
the static neighbour graph it builds from the coordinates: neither looks at the routing tree.  The seed is the answer only
when the routing path is the widest path, so the cases below edit states (through ``env.view``) into the regimes where it is
not: a low-lifetime relay near the base station, deaths the tree does not know yet, stale levels long after Network.operate
has stopped, alive nodes cut off from the base station, ``energyCS == 0`` (lifetime ``+inf``) and lifetime 0, and chains of
576 and 1152 nodes whose seed is wrong from one end to the other.  Every value is compared bit for bit: after one division
per node only comparisons, minima and maxima are involved.

The host build runs every environment on one lane, so the relaxation's rounds across warps and the atomics run on the GPU
only (``-m gpu``, 32, 64 and 128 threads).  Each case counts, on the host from the views, how often it reached its regime
(nodes whose answer exceeds their routing-path bottleneck, alive nodes with a dead receiver, alive ``cs == 0`` nodes, the
relaxation rounds a chain needs) and fails if too few states did."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, Scenario, synthetic
from multi_agent_rl_wrsn_b200.scenario import DEFAULT_MC, DEFAULT_NODE_PHY
from oracle import fitness_oracle as fo
from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO, golden, golden_names, scenario_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
SENTINEL = -7.25


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


def _np(t):
    return t.detach().cpu().numpy().copy()


_SCEN = {}


def field(N, seed):
    if (N, seed) not in _SCEN:
        _SCEN[(N, seed)] = synthetic(num_nodes=N, num_targets=N, seed=seed, num_gateways=3)
    return _SCEN[(N, seed)]


def hairpin(N):
    """A chain of N (even) nodes 72 m apart, folded once: rail A runs out from 45 m below the base station, rail B comes back to
    45 m above it, and the two rails meet only at the far end (their last nodes 70 m apart; everything else on the other rail is
    more than the 80.1 m communication range away).  Node 0 (A's first) and node N - 1 (B's first) are the only direct nodes.
    One target 5 m beside every node, covered by that node alone."""
    half = N // 2
    bs = np.array([100.0, 500.0])
    xy = np.zeros((N, 2))
    for i in range(N):
        j, side = (i, -1.0) if i < half else (N - 1 - i, 1.0)
        xy[i] = bs + (72.0 * j, side * (35.0 if j == half - 1 else 45.0))
    return Scenario(nodes=xy, targets=xy + (3.0, 4.0), base_station=bs, node_phy_spe=dict(DEFAULT_NODE_PHY), seed=0,
                    max_time=604800.0, name="hairpin%d" % N)


# ------------------------------------------------------------------ the comparison and its witnesses
_GRAPH = {}


def graph_of(sc):
    key = id(sc)
    if key not in _GRAPH:
        spe = sc.node_phy_spe
        _GRAPH[key] = (sc, fo.static_graph(sc.nodes, sc.targets, sc.base_station, float(spe["com_range"]), float(spe["sen_range"])))
    return _GRAPH[key][1]


def routing_seed(parent, status, lt):
    """do_fitness's starting point, restated: per alive node the bottleneck of its routing path (receiver by receiver to the
    base station), -1 where the walk meets a dead receiver or a node without one."""
    N = len(parent)
    seed = np.full(N, -1.0)
    for i in np.nonzero(status == 1)[0]:
        mn, h, hops = lt[i], int(parent[i]), 0
        while h >= 0 and hops < N:
            if status[h] != 1:
                h = -1
                break
            mn = min(mn, lt[h])
            h, hops = int(parent[h]), hops + 1
        if h == -2:
            seed[i] = mn
    return seed


def relaxation_rounds(g, lt, seed, parent):
    """Rounds of a synchronous (every node reads the previous round) pull relaxation from `seed` to its fixpoint: how far the
    answer has to travel against the routing tree."""
    alive = ~np.isnan(lt)
    src = np.concatenate([g["nbr"][i] for i in range(len(lt))] + [np.zeros(0, np.int64)]).astype(np.int64)
    dst = np.repeat(np.arange(len(lt)), [len(x) for x in g["nbr"]])
    keep = alive[src] & alive[dst] & (parent[dst] != -2)
    src, dst = src[keep], dst[keep]
    v, rounds = seed.copy(), 0
    while True:
        best = np.full(len(lt), -1.0)
        np.maximum.at(best, dst, v[src])
        nv = np.where(best >= 0.0, np.minimum(lt, best), -1.0)
        nv = np.where(nv > v, nv, v)
        if np.array_equal(nv, v):
            return rounds
        v, rounds = nv, rounds + 1


class Witness:
    """Per compared state: nodes whose answer exceeds their routing-path seed, alive nodes whose receiver is dead, alive nodes
    cut off from the base station, alive cs == 0 nodes, lifetime-0 nodes, +inf / 0 targets, +inf minima, relaxation rounds."""
    KEYS = ("wider", "dead_parent", "cut_off", "cs0", "life0", "inf_targets", "zero_targets", "inf_min", "rounds")

    def __init__(self):
        self.n = 0
        self.sum = dict.fromkeys(self.KEYS, 0)
        self.states = dict.fromkeys(self.KEYS, 0)
        self.max_rounds = 0

    def add(self, g, lt, node, seed, parent, status, per_target, mn, rounds):
        alive = status == 1
        reached = ~np.isnan(node)
        par_dead = alive & (parent >= 0) & (status[np.maximum(parent, 0)] != 1)
        cnt = dict(wider=int((reached & (node > seed)).sum()), dead_parent=int(par_dead.sum()), cut_off=int((alive & ~reached).sum()),
                   cs0=int((alive & np.isinf(lt)).sum()), life0=int((alive & (lt == 0.0)).sum()),
                   inf_targets=int(np.isinf(per_target).sum()), zero_targets=int((per_target == 0.0).sum()),
                   inf_min=int(np.isinf(mn)), rounds=rounds)
        self.n += 1
        for k, v in cnt.items():
            self.sum[k] += v
            self.states[k] += int(v > 0)
        self.max_rounds = max(self.max_rounds, rounds)

    def __repr__(self):
        return "states %d; per key (total, states): %s; max rounds %d" % (
            self.n, ", ".join("%s %d/%d" % (k, self.sum[k], self.states[k]) for k in self.KEYS), self.max_rounds)


def device_fitness(env):
    """``wrsn_fitness`` straight into sentinel-filled buffers: (per-target [B, T], minimum [B]) on the host."""
    fit = torch.full((env.B, max(env.T, 1)), SENTINEL, dtype=torch.float64, device=env.device)
    mn = torch.full((env.B,), SENTINEL, dtype=torch.float64, device=env.device)
    env._call(env.L.wrsn_fitness, C.byref(env.dims), env.scen.data_ptr(), env.scen_id.data_ptr(), env.state.data_ptr(),
              fit.data_ptr(), mn.data_ptr(), env._stream())
    return _np(fit), _np(mn)


def check_fitness(env, w, rows=None, with_rounds=False):
    """Every row (or `rows`): the device's per-target fitness and minimum == the restatement's, bit for bit, on the row's own
    targets; the columns beyond them keep the sentinel.  Adds each row to the witness `w`."""
    fit, mn = device_fitness(env)
    energy, cs, status, parent = (_np(env.view(f)) for f in ("energy", "cs", "status", "parent"))
    sid = _np(env.scen_id)
    for b in range(env.B) if rows is None else rows:
        sc = env.scenarios[int(sid[b])]
        g, n, t = graph_of(sc), sc.N, sc.T
        thr = float(sc.node_phy_spe["threshold"])
        want_min, want, node = fo.fitness(g, energy[b][:n], cs[b][:n], status[b][:n], thr)
        tag = ("row", b)
        pc.assert_bits(fit[b][:t], want, tag, "per-target fitness")
        pc.assert_bits(mn[b], want_min, tag, "fitness minimum")
        assert (fit[b][t:] == SENTINEL).all(), (tag, "columns beyond the row's targets were written")
        lt = fo.lifetimes(energy[b][:n], cs[b][:n], status[b][:n], thr)
        par = parent[b][:n].astype(np.int64)
        seed = routing_seed(par, status[b][:n], lt)
        rounds = relaxation_rounds(g, lt, seed, par) if with_rounds else 0
        w.add(g, lt, node, seed, par, status[b][:n], want, want_min, rounds)
    return fit, mn


def _set(env, name, b, idx, value):
    v = env.view(name)
    v[b, torch.as_tensor(np.atleast_1d(idx), dtype=torch.long, device=env.device)] = value


# ------------------------------------------------------------------ 1. the restatement against the fixtures and the C oracle
@pytest.mark.parametrize("name", golden_names("ep_"))
def test_restatement_matches_golden_fitness_min(name):
    """The restatement on the reference's own node records reproduces the minimum the reference computed, at every request."""
    g = golden(name)
    sc = scenario_of(g)
    p = sc["par"]
    graph = fo.static_graph(sc["nodes"], sc["targets"], sc["bs"], p[2], p[3])
    n = int(g["n"])
    for i in range(n):
        mn, _, _ = fo.fitness(graph, g["energy"][i], g["cs"][i], g["status"][i], p[1])
        want = float(g["fitness_min"][i])
        if np.isfinite(want):
            np.testing.assert_allclose(mn, want, rtol=1e-12, err_msg=str((name, i)))
        else:
            assert mn == want, (name, i, mn, want)


@pytest.mark.parametrize("N,seed,R", [(60, 41, 27.0), (100, 42, 80.0), (150, 43, 27.0)])
def test_restatement_equals_c_oracle(N, seed, R):
    """The static graph and, at every request of a random episode, every target's value == orc_fitness, bit for bit."""
    sc = field(N, seed)
    spe = sc.node_phy_spe
    mc = dict(DEFAULT_MC, charging_range=R)
    o = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=3, mc=mc)
    graph = fo.static_graph(sc.nodes, sc.targets, sc.base_station, float(spe["com_range"]), float(spe["sen_range"]))
    st = o.static_graph()
    for i in range(N):
        assert np.array_equal(graph["nbr"][i], st["nbr_idx"][st["nbr_ptr"][i]:st["nbr_ptr"][i + 1]]), i
        assert np.array_equal(graph["cover"][i], st["tgt_idx"][st["tgt_ptr"][i]:st["tgt_ptr"][i + 1]]), i
    assert np.array_equal(graph["direct"], st["direct"] != 0)
    rng = np.random.default_rng(seed)
    r = o.reset(want_state=False)
    zero = checked = 0
    for k in range(80):
        nd = o.nodes()
        omin, ofit = o.fitness()
        mn, per_target, _ = fo.fitness(graph, nd["energy"], nd["cs"], nd["status"], float(spe["threshold"]))
        pc.assert_bits(per_target, ofit, k, "per-target fitness")
        pc.assert_bits(mn, omin, k, "fitness minimum")
        zero += int((ofit == 0).sum())
        checked += 1
        if r["raw_agent_id"] < 0 and r["raw_agent_id"] != -2:
            break
        a = rng.uniform(0, 1, 3)
        a[2] *= 0.3
        r = o.step(r["raw_agent_id"] if r["raw_agent_id"] >= 0 else None, a, want_state=False)
    assert checked >= 15 and zero > 0, (checked, zero)      # the episode ran on into deaths and uncovered targets


# ------------------------------------------------------------------ 2. the device against the restatement
THREADS = [cpu(0, id="cpu")] + [gpu(th, id="gpu-t%d" % th) for th in (32, 64, 128)]


def _env(scs, dev, threads, B, num_agent=3):
    env = BatchedWRSN(scs, num_agent=num_agent, num_envs=B, device=dev, threads=threads)
    env.reset()
    return env


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_real_states(dev, threads):
    """Rollouts on three 100-node fields under uniform actions, every row after every step, until most nodes have died."""
    env = _env([field(100, s) for s in (7, 8, 9)], dev, threads, B=6)
    rng = np.random.default_rng(threads)
    w = Witness()
    for k in range(60):
        check_fitness(env, w)
        a = rng.uniform(0, 1, (env.B, 3))
        a[:, 2] *= 0.3
        env.rollout_step(torch.as_tensor(a, device=env.device))
    assert w.n == 60 * env.B and w.states["wider"] >= 0.5 * w.n and w.states["cs0"] == w.n, w


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_low_bottleneck_near_the_base_station(dev, threads):
    """The relay with the most nodes routing through it gets a lifetime of 1e-3 s (then 0): its whole subtree's seed is that
    bottleneck, while most of those nodes have a wider path around it."""
    scs = [field(100, s) for s in (11, 12, 13, 14)]
    env = _env(scs, dev, threads, B=4)
    w = Witness()
    status, parent, cs = _np(env.view("status")), _np(env.view("parent")).astype(np.int64), _np(env.view("cs"))
    thr = float(scs[0].node_phy_spe["threshold"])
    relays = []
    for b in range(env.B):
        n = env.scenarios[int(env.scen_id[b])].N
        below = np.zeros(n, np.int64)
        for i in range(n):                               # nodes routing through each relay
            h = parent[b][i]
            while h >= 0:
                below[h] += 1
                h = parent[b][h]
        relay = int(np.argmax(below))
        _set(env, "energy", b, relay, thr + 1e-3 * cs[b][relay])
        relays.append(relay)
    check_fitness(env, w)
    for b in range(env.B):
        _set(env, "energy", b, relays[b], thr)
    check_fitness(env, w)
    assert w.states["wider"] == w.n and w.sum["wider"] >= 20 * w.n and w.states["life0"] == env.B, w


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_deaths_the_tree_does_not_know(dev, threads):
    """status set to 0 without a BFS: one relay per row, then every third relay — the routing walks end at dead receivers."""
    env = _env([field(100, s) for s in (21, 22, 23)], dev, threads, B=3)
    w = Witness()
    parent = _np(env.view("parent")).astype(np.int64)
    for b in range(env.B):
        relays = np.unique(parent[b][parent[b] >= 0])
        _set(env, "status", b, relays[len(relays) // 2], 0)
    check_fitness(env, w)
    for b in range(env.B):
        relays = np.unique(parent[b][parent[b] >= 0])
        _set(env, "status", b, relays[::3], 0)
    check_fitness(env, w)
    assert w.states["dead_parent"] == w.n and w.states["wider"] == w.n and w.states["cut_off"] >= 1, w


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_stale_levels_after_network_operate(dev, threads):
    """A pure network run far past the end of Network.operate (alive == 0): levels stay stale, later deaths re-route through
    them, and the direct nodes die first: the routing paths left are not the widest ones, and most nodes end up cut off."""
    sc = field(100, 31)
    env = BatchedWRSN(sc, num_agent=0, num_envs=1, device=dev, threads=threads)
    env.init_network(with_reward_process=False)
    w = Witness()
    t = 100.25
    while t < 40000.0:
        env.run_until(t)
        check_fitness(env, w)
        t += 601.0
    assert float(_np(env.hdr("NET_ON"))[0]) == 0.0
    assert w.states["wider"] >= 3 and w.states["cut_off"] >= 0.5 * w.n, w


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_cut_off_nodes(dev, threads):
    """A band of dead nodes (without a BFS) wider than the communication range across the whole field, 150 m beside the base
    station: the alive nodes beyond it are cut off and the targets only they cover get 0.  In the last row every direct node
    is dead as well, and the minimum is 0."""
    scs = [field(100, s) for s in (41, 42)]
    env = _env(scs, dev, threads, B=3)
    w = Witness()
    for b in range(env.B):
        sc = env.scenarios[int(env.scen_id[b])]
        dx = sc.nodes[:, 0] - sc.base_station[0]
        band = np.nonzero((dx > 150.0) & (dx < 240.0))[0]
        if b == 2:
            band = np.union1d(band, np.nonzero(env.statics[int(env.scen_id[b])]["direct"][:sc.N])[0])
        _set(env, "status", b, band, 0)
    fit, mn = check_fitness(env, w)
    assert w.states["cut_off"] == w.n and w.sum["cut_off"] >= 3 * 20 and w.states["zero_targets"] == w.n and mn[2] == 0.0, w


@pytest.mark.parametrize("dev,threads", THREADS, indirect=["dev"])
def test_infinite_and_zero_lifetimes(dev, threads):
    """energyCS == 0 on alive nodes: on every node of row 0 (every target and the minimum +inf), on the direct nodes only in row
    1 (+inf bottlenecks at the root, finite values further out), on every other node in row 2 together with one lifetime of
    exactly 0 (energy == threshold)."""
    sc = field(100, 51)
    env = _env([sc], dev, threads, B=3)
    w = Witness()
    st = env.statics[0]
    thr = float(sc.node_phy_spe["threshold"])
    _set(env, "cs", 0, np.arange(sc.N), 0.0)
    _set(env, "cs", 1, np.nonzero(st["direct"][:sc.N])[0], 0.0)
    _set(env, "cs", 2, np.arange(0, sc.N, 2), 0.0)
    _set(env, "energy", 2, 3, thr)
    fit, mn = check_fitness(env, w)
    assert np.isinf(mn[0]) and np.isinf(fit[0][:sc.T]).all() and np.isfinite(mn[1])
    assert w.states["cs0"] == 3 and w.states["inf_targets"] >= 2 and w.sum["inf_min"] == 1 and w.sum["life0"] == 1, w


CHAIN_CASES = [cpu(576, 0, id="cpu-N576"), cpu(1152, 0, id="cpu-N1152")] + \
              [gpu(N, th, id="gpu-N%d-t%d" % (N, th)) for N, th in ((128, 32), (576, 64), (576, 128), (1152, 128))]


@pytest.mark.parametrize("dev,N,threads", CHAIN_CASES, indirect=["dev"])
def test_deep_chains(dev, N, threads):
    """The folded chain with its first node dead (no BFS): every node of rail A routes to that node, so its seed is -1, and its
    answer comes around the fold over the whole of rail B — N / 2 hops against the routing tree, relaxed round by round (on
    the GPU across every warp of the row).  Then the same with one low-lifetime node on rail B, which the answers of rail A
    must all take on."""
    env = _env(hairpin(N), dev, threads, B=2, num_agent=1)
    assert int(_np(env.alive)[0]) == 1 and (_np(env.view("status"))[:, :N] == 1).all()
    w = Witness()
    _set(env, "status", 0, 0, 0)
    _set(env, "status", 1, 0, 0)
    cs = _np(env.view("cs"))
    thr = float(DEFAULT_NODE_PHY["threshold"])
    k = N - 1 - N // 4                                   # halfway along rail B
    _set(env, "energy", 1, k, thr + 0.5 * cs[1][k])
    check_fitness(env, w, with_rounds=True)
    assert w.sum["wider"] >= 2 * (N // 2 - 1) and w.max_rounds >= N // 2 - 2, w


# ------------------------------------------------------------------ 3. a mixed-size batch
@pytest.mark.parametrize("dev,threads", [cpu(0, id="cpu"), gpu(64, id="gpu-t64"), gpu(128, id="gpu-t128")], indirect=["dev"])
def test_mixed_size_batch(dev, threads):
    """Rows of 50, 100 and 150 nodes (as many targets) in one batch, real and edited states: every row's own columns == the
    restatement and the columns beyond its target count keep the caller's sentinel (include/wrsn_b200.h)."""
    scs = [field(50, 61), field(150, 62), field(100, 63)]
    env = _env(scs, dev, threads, B=6)
    w = Witness()
    rng = np.random.default_rng(6)
    for k in range(30):
        check_fitness(env, w)
        a = rng.uniform(0, 1, (env.B, 3))
        a[:, 2] *= 0.2
        env.rollout_step(torch.as_tensor(a, device=env.device))
    parent = _np(env.view("parent")).astype(np.int64)
    for b in range(env.B):
        relays = np.unique(parent[b][parent[b] >= 0])
        if len(relays):
            _set(env, "status", b, relays[::4], 0)
        _set(env, "cs", b, np.arange(b, env.N, 7), 0.0)
    check_fitness(env, w)
    assert w.n == 31 * env.B and w.states["dead_parent"] >= 4 and w.states["cs0"] >= 4, w


# ------------------------------------------------------------------ 4. lazy charger spans, replayed several slots at a time
def _moving(env):
    """Per row: chargers that are alive and not at their destination."""
    at = (env.mc("X") == env.mc("CPA0")) & (env.mc("Y") == env.mc("CPA1"))
    return ((env.mc("STATUS") != 0) & ~at).sum(1).cpu().numpy()


LAZY_CASES = [cpu(300, 0, 2, 25, id="cpu-N300"), gpu(100, 32, 8, 40, id="gpu-N100-t32"), gpu(300, 64, 8, 40, id="gpu-N300-t64"),
              gpu(500, 128, 4, 40, id="gpu-N500-t128")]


@pytest.mark.parametrize("dev,N,threads,rows,steps", LAZY_CASES, indirect=["dev"])
def test_sixteen_moving_chargers_vs_oracle(dev, N, threads, rows, steps):
    """16 chargers on fields of up to 2.2 km, short charges (at most 1 % of the longest) and actions drawn from [-0.25, 1.25]
    (clipped): most of the time many chargers are on long moves at once, whose seconds the engine replays lazily — on the GPU
    one thread per slot (catch_up_many) when update_reward reads their positions.  Every request against the oracle, the
    chargers' X / Y among everything else bit for bit.  Witness, per row and step: the process slots that stayed lazy across
    the step while their owed insertion counters grew (spans replayed without waking: catch_up_many's work), and NLAZY."""
    sc = synthetic(num_nodes=N, num_targets=N, seed=N + 5, num_gateways=max(3, N // 40))
    moving, multi, prev = [], [], {}

    def probe(env, live):
        E = env.E
        lazy = env.view("proc").view(torch.int32)[:, :, E["WRSN_PRI_LAZY"]].cpu().numpy() != 0
        owed = _np(env.view("proc")[:, :, E["WRSN_PR_OWED"]])
        nlazy = _np(env.hdr("NLAZY"))
        if prev:
            replayed = (prev["lazy"] & lazy & (owed > prev["owed"])).sum(1)          # slots replayed in place during the step
            grew = nlazy > prev["nlazy"]
            multi.extend((replayed[live] >= 2) & grew[live])
        prev.update(lazy=lazy, owed=owed, nlazy=nlazy)
        moving.extend(_moving(env)[live].tolist())
    n_dec, cnt = pc.check_vs_oracle(sc, dev, num_envs=rows, steps=steps, seed=N, num_agent=16, scale2=0.01, threads=threads,
                                    probe=probe, spread=0.25)
    moving, multi = np.array(moving), np.array(multi)
    assert n_dec >= rows * steps // 2, n_dec
    assert (moving >= 8).mean() >= 0.5 and cnt["lazy_spans"] >= 50 * rows * steps, (np.bincount(moving), cnt)
    assert multi.sum() >= 0.25 * len(multi), (int(multi.sum()), len(multi))


# ------------------------------------------------------------------ 5. energyCS where a relay's per-tick log is long
def test_oracle_send_cost_is_libm_pow():
    """Node.send_package's ``d ** 2`` is a libm pow call in the reference and in scenario.py's e_send table; a literal
    pow(d, 2.0) in C is folded into d * d, which differs from glibc's pow by one ulp for some d.  On the 300-node field below
    node 93 relays 8 packets after the death at 663.5 s and its per-tick log (an 11-term sum of e_send / e_receive) then ends
    2 ulp apart unless the oracle calls pow too: energyCS, the mean of those logs, must agree bit for bit with the engine's
    table through that re-route (the energies alone do not show it)."""
    import math
    from multi_agent_rl_wrsn_b200.scenario import _e_send
    sc = field_cs()
    helpers.use_host_build()
    try:
        env = BatchedWRSN(sc, num_agent=0, num_envs=1, device="cpu")
        env.init_network(with_reward_process=False)
        o = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=0)
        o.start_network_only()
        t = 600.25
        env.run_until(t)
        o.run_until(t)
        while t < 700.0:
            env.run_until(t)
            o.run_until(t)
            nd = o.nodes()
            assert np.array_equal(_np(env.view("status"))[0], nd["status"]), t
            pc.assert_bits(_np(env.view("cs"))[0], nd["cs"], t, "node cs")
            pc.assert_bits(_np(env.view("energy"))[0], nd["energy"], t, "node energy")
            t += 0.5
        assert int((nd["status"] == 0).sum()) >= 1 and int(_np(env.view("naft"))[0][93]) == 8
    finally:
        helpers.use_cuda_build_lazy()
    d = 61.71026423045482                                  # node 93 -> its receiver 193 after the re-route
    assert _e_send(d, sc.node_phy_spe) == float((sc.node_phy_spe["et"] + sc.node_phy_spe["efs"] * math.pow(d, 2.0))
                                                * sc.node_phy_spe["package_size"])


def field_cs():
    return synthetic(num_nodes=300, num_targets=300, seed=300, num_gateways=7)


CS_CASES = [cpu(0, id="cpu")] + [gpu(th, id="gpu-t%d" % th) for th in (64, 128)]


@pytest.mark.parametrize("dev,threads", CS_CASES, indirect=["dev"])
def test_relay_logs_after_reroutes_vs_oracle(dev, threads):
    """The configurations where energyCS first left the oracle's (a relay's log 2 ulp off after a re-route; then the decaying
    mean of an alive node on the other side of 0 and the exclusive reward 1e-3 off): the dense fuzz seed 7017 (173 nodes, 8
    chargers) and the 1152-node field, every row at every request bit for bit."""
    from tests.test_crowded import fuzz_case
    sc, M, R, scale2, steps = fuzz_case(7017)
    n_dec, _ = pc.check_vs_oracle(sc, dev, num_envs=3, steps=steps, seed=7017, num_agent=M, mc=dict(DEFAULT_MC, charging_range=R),
                                  scale2=scale2, threads=threads)
    assert n_dec >= 40, n_dec
    big = synthetic(num_nodes=1152, num_targets=1152, seed=1152, num_gateways=1152 // 40)
    n_dec, cnt = pc.check_vs_oracle(big, dev, num_envs=2, steps=25, seed=9, num_agent=3, scale2=0.05,
                                    threads=max(threads, 128) if threads else 0)
    assert n_dec >= 10 and cnt["bfs"] >= 10, (n_dec, cnt)
