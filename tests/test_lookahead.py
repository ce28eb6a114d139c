"""The lookahead planner: ranked candidates (BatchedWRSN.heuristic_candidates, wrsn_heuristic_candidates), branch rollouts
(BatchedWRSN.lookahead) and LookaheadController.

The candidate order is checked bit for bit against ``rank`` below, a numpy restatement over the state views built on
oracle/heuristic_oracle.py, on the host build of the kernel source and (``-m gpu``) on k_heuristic_candidates, which must also
equal the host build byte for byte.  Lookahead values are checked bit for bit against replays of each branch driven by hand in
a fresh batch.  Each regime a case is meant to reach is counted, and the case fails below a floor."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, EnvSnapshot, HeuristicController, LookaheadController, _lib, evaluate, rollout, synthetic
from oracle import heuristic_oracle as ho
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO, golden, mc_dict_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
GOLDEN3 = ("ep_basic_n50", "ep_full_n100", "ep_full_n200")      # 82 / 98 / 132 nodes
W_RANDOM = (1.0, 1.0, -10.0, 1.0)
KINDS = ho.KINDS
WIDTHS = (1, 3, 8, 32)
SENTINEL = 7.25
NODE_SENTINEL = -7


@pytest.fixture(scope="module")
def emu_built():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)


@pytest.fixture
def host(emu_built):
    helpers.use_host_build()
    yield "cpu"
    helpers.use_cuda_build_lazy()


def _np(t):
    return t.detach().cpu().numpy().copy()


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.int64)


def _scenarios(synth=True):
    gs = [golden(n) for n in GOLDEN3]
    return [pc.sc_from_golden(g) for g in gs] + ([synthetic(100, 100, seed=1000)] if synth else []), mc_dict_of(gs[0])


def _mixed(B=8, device="cpu", synth=True, **kw):
    scs, mc = _scenarios(synth)
    return BatchedWRSN(scs, num_agent=kw.pop("num_agent", 3), mc_type=mc, num_envs=B, device=device, **kw)


# ------------------------------------------------------------------ the restatement of the order
def rank(kind, a, n, x, y, energy, cs, status, mc_x, mc_y, mc_status, mc_dest_x, mc_dest_y, par):
    """Every candidate of heuristic_oracle.choose's candidate set, in the rule's order: np.lexsort over (id, key, class) — class 0
    the urgent nodes of nearest_urgent keyed by the distance from charger a, class 1 the rest keyed by the lifetime."""
    x, y = np.asarray(x, np.float64)[:n], np.asarray(y, np.float64)[:n]
    energy, cs = np.asarray(energy, np.float64)[:n], np.asarray(cs, np.float64)[:n]
    alive = np.asarray(status)[:n] == 1
    with np.errstate(divide="ignore", invalid="ignore"):
        life = np.where(cs <= 0.0, np.inf, (energy - par["THR"]) / cs)
    claimed = np.zeros(n, bool)
    for j in range(len(mc_x)):
        if j != a and mc_status[j] != 0:
            claimed |= ho.euclid(x, y, mc_dest_x[j], mc_dest_y[j]) <= par["MC_R"]
    cand = alive & ~claimed
    if not cand.any():
        cand = alive
    c = np.nonzero(cand)[0]
    cls = np.ones(c.size, np.int64)
    key = life[c].copy()
    if kind == "nearest_urgent":
        urgent = life[c] < par["MTM"] + par["CTM"]
        cls[urgent] = 0
        key[urgent] = ho.euclid(mc_x[a], mc_y[a], x[c[urgent]], y[c[urgent]])
    return c[np.lexsort((c, key, cls))]


def _rows(env):
    E = env.E
    energy, cs, status, mc = _np(env.view("energy")), _np(env.view("cs")), _np(env.view("status")), _np(env.view("mc"))
    sid = _np(env.scen_id)
    for b in range(env.B):
        st = env.statics[int(sid[b])]
        m = mc[b, :env.M]
        yield b, dict(n=st["N"], x=np.asarray(st["x"], np.float64), y=np.asarray(st["y"], np.float64), energy=energy[b], cs=cs[b],
                      status=status[b], mc_x=m[:, E["WRSN_MC_X"]], mc_y=m[:, E["WRSN_MC_Y"]], mc_status=m[:, E["WRSN_MC_STATUS"]],
                      mc_dest_x=m[:, E["WRSN_MC_CPA0"]], mc_dest_y=m[:, E["WRSN_MC_CPA1"]], par=st["par"])


def oracle(env, kind, K, agent_id=None):
    """The restatement's actions [B, K, 3] and nodes [B, K] (rows without a deciding charger: the sentinels), and how many
    candidates each row has (-1 without a decider)."""
    aid = _np(env.req.agent_id if agent_id is None else torch.as_tensor(agent_id))
    act, node = np.full((env.B, K, 3), SENTINEL), np.full((env.B, K), NODE_SENTINEL, np.int32)
    count = np.full(env.B, -1)
    for b, r in _rows(env):
        a = int(aid[b])
        if a < 0 or a >= env.M:
            continue
        order = rank(kind, a, r["n"], r["x"], r["y"], r["energy"], r["cs"], r["status"], r["mc_x"], r["mc_y"], r["mc_status"],
                     r["mc_dest_x"], r["mc_dest_y"], r["par"])
        count[b] = order.size
        node[b] = -1
        node[b, :min(K, order.size)] = order[:K]
        first = int(order[0]) if order.size else -1
        for k in range(K):
            i = int(node[b, k]) if node[b, k] >= 0 else first
            act[b, k] = ho.action(i, a, r["x"], r["y"], r["energy"], r["mc_x"], r["mc_y"], r["par"])
    return act, node, count


def check_candidates(env, kind, K, agent_id=None):
    """heuristic_candidates == the restatement bit for bit, slot 0 == heuristic_action byte for byte, and rows without a
    deciding charger keep the sentinels.  -> the candidate count of every row (-1: no decider)."""
    out = torch.full((env.B, K, 3), SENTINEL, dtype=torch.float64, device=env.device)
    nd = torch.full((env.B, K), NODE_SENTINEL, dtype=torch.int32, device=env.device)
    got_a, got_n = env.heuristic_candidates(kind, K, agent_id=agent_id, out=out, node=nd)
    got_a, got_n = _np(got_a), _np(got_n)
    want_a, want_n, count = oracle(env, kind, K, agent_id)
    assert np.array_equal(got_n, want_n), (kind, K, np.nonzero((got_n != want_n).any(1))[0][:8])
    assert np.array_equal(_bits(got_a), _bits(want_a)), (kind, K, np.nonzero((_bits(got_a) != _bits(want_a)).any((1, 2)))[0][:8])
    h = _np(env.heuristic_action(kind, agent_id=agent_id, out=torch.full((env.B, 3), SENTINEL, dtype=torch.float64, device=env.device)))
    assert np.array_equal(_bits(got_a[:, 0]), _bits(h)), (kind, K)
    return count


def check_all(env, kinds=KINDS, widths=WIDTHS):
    """check_candidates for every kind and width, with the request's decider and with every charger as the decider."""
    counts = []
    for kind in kinds:
        for K in widths:
            counts.append(check_candidates(env, kind, K))
            for a in range(env.M):
                counts.append(check_candidates(env, kind, K, torch.full((env.B,), a, dtype=torch.int32, device=env.device)))
    return np.concatenate(counts)


# ------------------------------------------------------------------ 1. candidates: host build == restatement
def test_mixed_batch_candidates_equal_the_restatement(host):
    env = _mixed(B=8)
    env.reset()
    check_all(env)
    acts = np.random.default_rng(4).uniform(0.0, 1.0, size=(40, env.B, 3))
    acts[..., 2] *= 0.1
    for t in range(40):
        env.rollout_step(torch.as_tensor(acts[t]))
    assert (_np(env.req.stats)[:, 0] >= 40).all()
    counts = check_all(env)
    assert (counts >= 32).sum() >= 8                                  # rows that fill every slot at K = 32


# ------------------------------------------------------------------ 2. candidates on edited states
def _set_mc(env, b, j, **fields):
    mc = env.view("mc")
    for k, v in fields.items():
        mc[b, j, env.E["WRSN_MC_" + k]] = v


def _xy(env, b, i):
    st = env.statics[int(env.scen_id[b])]
    return float(st["x"][i]), float(st["y"][i])


def _clear_claims(env, b):
    for j in range(env.M):
        _set_mc(env, b, j, CPA0=-1e6, CPA1=-1e6)


def _edit_env(B=3):
    env = _mixed(B=B, synth=False)                                    # rows 82 / 98 / 132 nodes, N = 132
    env.reset()
    for b in range(B):
        _clear_claims(env, b)
    return env


def test_candidates_on_edited_states(host):
    few = 0
    # ties: equal lifetimes, nodes without traffic (key +inf), and equal distances from the decider
    env = _edit_env()
    par = env.statics[0]["par"]
    horizon = par["MTM"] + par["CTM"]
    e, cs = env.view("energy"), env.view("cs")
    cs[0, :82] = 1.0
    e[0, :82] = par["THR"] + 3.0 * horizon
    e[0, [31, 9, 20, 40]] = par["THR"] + 2.0 * horizon               # equal and lowest, not urgent
    cs[0, [5, 6, 7]] = 0.0
    e[1, [3, 11, 17]] = env.statics[1]["par"]["THR"] + 0.5 * horizon  # urgent in row 1
    x3, y3 = _xy(env, 1, 3)
    _set_mc(env, 1, 0, X=x3, Y=y3)
    for b in range(3):
        e[b, 12] = e[b, 13] = env.statics[int(env.scen_id[b])]["par"]["THR"] + 0.1 * horizon   # urgent, distance ties below
    xa, ya = _xy(env, 2, 12)
    xb, yb = _xy(env, 2, 13)
    _set_mc(env, 2, 0, X=(xa + xb) / 2.0, Y=(ya + yb) / 2.0)
    few += (check_all(env) < 32).sum()
    order = _np(env.heuristic_candidates("min_lifetime", 32, agent_id=torch.zeros(3, dtype=torch.int32))[1])[0]
    assert order[:6].tolist() == [12, 13, 9, 20, 31, 40] and order[6:].tolist() == [i for i in range(82) if i not in (5, 6, 7, 9, 12, 13, 20, 31, 40)][:26]
    # every alive node claimed; fewer candidates than slots; a dead charger claims nothing
    env = _edit_env()
    st = env.view("status")
    st[0, :] = 0
    st[0, [7, 12, 30]] = 1
    for j, i in ((1, 7), (2, 12)):
        x, y = _xy(env, 0, i)
        _set_mc(env, 0, j, STATUS=1.0, CPA0=x, CPA1=y)
    c = check_all(env)
    few += (c < 32).sum()
    assert _np(env.heuristic_candidates("min_lifetime", 3, agent_id=torch.zeros(3, dtype=torch.int32))[1])[0].tolist()[1:] == [-1, -1]
    st[0, 30] = 0                                                     # now only claimed nodes are alive: both come back
    c = check_all(env)
    nodes = _np(env.heuristic_candidates("min_lifetime", 4, agent_id=torch.zeros(3, dtype=torch.int32))[1])[0]
    assert sorted(nodes[:2].tolist()) == [7, 12] and nodes[2:].tolist() == [-1, -1]
    _set_mc(env, 0, 2, STATUS=0.0)                                    # dead: 12 is no longer claimed, 7 still is
    assert _np(env.heuristic_candidates("min_lifetime", 4, agent_id=torch.zeros(3, dtype=torch.int32))[1])[0].tolist() == [12, -1, -1, -1]
    few += (check_all(env) < 32).sum()
    # no node alive: every slot -1, every action the stay action
    st[0, :] = 0
    check_all(env)
    act, nodes = env.heuristic_candidates("nearest_urgent", 5, agent_id=torch.zeros(3, dtype=torch.int32))
    assert _np(nodes)[0].tolist() == [-1] * 5 and (_np(act)[0] == _np(act)[0, :1]).all() and _np(act)[0, 0, 2] == 0.0
    # padding nodes of the smaller scenarios alive and about to die: never listed
    env = _edit_env()
    for b in (0, 1):
        n = int(env.num_nodes[b])
        env.view("status")[b, n:] = 1
        env.view("energy")[b, n:] = env.statics[int(env.scen_id[b])]["par"]["THR"] + 1e-6
        env.view("cs")[b, n:] = 1.0
    check_all(env)
    nodes = _np(env.heuristic_candidates("min_lifetime", 32, agent_id=torch.zeros(3, dtype=torch.int32))[1])
    assert (nodes[0] < 82).all() and (nodes[1] < 98).all()
    assert few >= 20


def test_rows_without_a_decider_keep_the_sentinels(host):
    env = _mixed(B=6, synth=False)
    env.reset()
    aid = torch.tensor([-1, 0, -4, 2, -2, 1], dtype=torch.int32)
    for kind in KINDS:
        for K in WIDTHS:
            count = check_candidates(env, kind, K, aid)
            assert (count[[0, 2, 4]] == -1).all() and (count[[1, 3, 5]] > 0).all()


# ------------------------------------------------------------------ refusals
@pytest.fixture(scope="module")
def cuda_so():
    import __graft_entry__ as g
    g.build()
    return ctypes.CDLL(_lib.LIB_PATH)


def test_refusals_equal_in_both_libraries(cuda_so, emu_built):
    libs = [_lib._bind(cuda_so), _lib._bind(ctypes.CDLL(os.path.join(EMU_DIR, "libwrsn_emu.so")))]

    def dims(L, finalize=True):
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = 2, 100, 100, 3, 100, 600, 200, 1
        if finalize:
            assert L.wrsn_dims_finalize(ctypes.byref(d)) == 0
        return d

    big = dims(libs[0])
    arrays = dict(scen=np.zeros(big.scen_bytes, np.uint8), scen_id=np.zeros(2, np.int32), state=np.zeros(big.state_bytes * 2, np.uint8),
                  agent=np.full(2, -1, np.int32), action=np.zeros(2 * 33 * 3, np.float64), node=np.zeros(2 * 33, np.int32))

    def call(L, d, null=None, kind=0, K=4):
        p = {k: (None if k == null else a.ctypes.data) for k, a in arrays.items()}
        rc = L.wrsn_heuristic_candidates(ctypes.byref(d), p["scen"], p["scen_id"], p["state"], p["agent"], kind, K, p["action"],
                                         p["node"], None)
        return rc, L.wrsn_last_error()

    cases = [(dict(finalize=False), {}, b"dims not finalized"), ({}, dict(null="action"), b"NULL argument"),
             ({}, dict(null="node"), b"NULL argument"), ({}, dict(null="agent"), b"NULL argument"),
             ({}, dict(kind=-1), b"heuristic kind -1"), ({}, dict(kind=2), b"heuristic kind 2"),
             ({}, dict(K=0), b"K = 0 candidates: 1 to 32"), ({}, dict(K=33), b"K = 33 candidates: 1 to 32"),
             ({}, dict(K=-5), b"K = -5 candidates")]
    for dkw, ckw, msg in cases:
        got = [call(L, dims(L, **dkw), **ckw) for L in libs]
        assert got[0] == got[1], (dkw, ckw, got)
        assert got[0][0] == -1 and msg in got[0][1], (dkw, ckw, got)
    for K in (1, 32):                                                 # the bounds themselves are accepted (the host build
        assert call(libs[1], dims(libs[1]), K=K)[0] == 0              # here: the CUDA library's launch needs a device)


def test_python_refusals(host):
    env = _mixed(B=2, synth=False)
    env.reset()
    for w in (0, 33):
        with pytest.raises(ValueError, match="width"):
            env.heuristic_candidates("min_lifetime", w)
    with pytest.raises(ValueError, match="kind"):
        env.heuristic_candidates("farthest_first", 4)
    with pytest.raises(ValueError, match="node"):
        env.heuristic_candidates("min_lifetime", 4, node=torch.zeros((2, 4), dtype=torch.int64))
    cand = torch.zeros((2, 4, 3), dtype=torch.float64)
    with pytest.raises(ValueError, match="candidates"):
        env.lookahead(cand.float(), 2)
    with pytest.raises(ValueError, match="rollout_kind"):
        env.lookahead(cand, 2, "random")
    with pytest.raises(ValueError, match="valid"):
        env.lookahead(cand, 2, valid=torch.ones((2, 3), dtype=torch.bool))
    with pytest.raises(ValueError, match="charge_levels"):
        LookaheadController(charge_levels=(1.5,))


# ------------------------------------------------------------------ 3. lookahead == replays driven by hand
def _record(env):
    """Everything lookahead must leave unchanged: the state records, scen_id and the request record."""
    q = env.req
    return [_np(x) for x in (env.state, env.scen_id, q.agent_id, q.terminal, q.reward, q.now, q.action, q.detail, q.flags, q.stats,
                             q.sticky)]


def replay(env, cand, valid, horizon, kind, make):
    """The value of every (row, slot) of ``env``, computed independently of lookahead: the rows are saved with snapshot and
    restored, at permuted positions, into a fresh batch of another size (``make(B)``), which is then driven request by request:
    the candidate for the deciding charger, then the rule until `horizon` more decisions are made or the episode ends; the
    rewards of the requests after each step are added in order on the host.  -> (values [B, K], branches that ended inside
    the horizon, branch steps that continued a step in flight)."""
    B, K = cand.shape[:2]
    aid0 = _np(env.req.agent_id)
    pairs = [(b, k) for b in range(B) for k in range(K) if aid0[b] >= 0 and valid[b, k]]
    vals = np.where(aid0[:, None] >= 0, np.where(valid, 0.0, -np.inf), np.nan)
    if not pairs:
        return vals, 0, 0
    R = len(pairs) + 5
    fresh = make(R)
    fresh.reset()
    perm = np.random.default_rng(len(pairs)).permutation(R)[:len(pairs)]
    snap = env.snapshot(rows=[b for b, _ in pairs])
    fresh.restore(snap, rows=perm)
    ret = {p: 0.0 for p in pairs}
    dec = {p: 0 for p in pairs}
    going = {p: True for p in pairs}
    ended = inflight = 0
    first = True
    while any(going.values()):
        aid = _np(fresh.req.agent_id)
        agent = np.full(R, -1, np.int32)
        act = np.zeros((R, 3))
        mask = np.zeros(R, bool)
        rule = _np(fresh.heuristic_action(kind))
        for p, r in zip(pairs, perm):
            if not going[p]:
                continue
            a = int(aid[r])
            if a == -1:
                going[p] = False
                ended += dec[p] < horizon + 1
                continue
            if a != -4 and dec[p] >= horizon + 1:
                going[p] = False
                continue
            mask[r] = True
            inflight += a == -4
            agent[r] = max(a, -1)
            act[r] = _np(cand[p[0], p[1]]) if first else rule[r]
            dec[p] += a >= 0
        if not mask.any():
            break
        first = False
        fresh.step(torch.as_tensor(agent, device=fresh.device), torch.as_tensor(act, device=fresh.device), mask=torch.as_tensor(mask, device=fresh.device))
        rew = _np(fresh.req.reward)
        for p, r in zip(pairs, perm):
            if mask[r]:
                x = float(rew[r])
                ret[p] += 0.0 if x != x else x
    fresh.raise_on_error()
    for (b, k), v in ret.items():
        vals[b, k] = v
    return vals, ended, inflight


def check_lookahead(env, cand, valid, horizon, kind, make):
    before = _record(env)
    got = _np(env.lookahead(cand, horizon, kind, valid))
    after = _record(env)
    for x, y in zip(before, after):
        assert x.tobytes() == y.tobytes()
    want, ended, inflight = replay(env, cand, _np(valid), horizon, kind, make)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(_bits(np.nan_to_num(got, nan=0.0)), _bits(np.nan_to_num(want, nan=0.0))), (got, want)
    return got, ended, inflight


def _short_lived():
    """A small network whose nodes start barely above threshold: it dies after a few decisions."""
    from multi_agent_rl_wrsn_b200.scenario import DEFAULT_NODE_PHY
    spe = dict(DEFAULT_NODE_PHY)
    spe["capacity"] = spe["threshold"] * 1.05
    return synthetic(30, 30, seed=7, node_phy_spe=spe)


@pytest.mark.parametrize("budget", [0, 60])
def test_lookahead_equals_replays(host, budget):
    env = _mixed(B=4, step_budget=budget)
    make = lambda R: _mixed(B=R, step_budget=budget)              # noqa: E731
    env.reset()
    rng = np.random.default_rng(10 + budget)
    for t in range(40):                                               # with a budget: until a row is in flight
        env.rollout_step(torch.as_tensor(rng.uniform(0.0, 1.0, size=(4, 3))))
        if t >= 5 and (not budget or (_np(env.req.agent_id) == -4).any()):
            break
    K, unequal, missing, inflight = 3, 0, 0, 0
    for kind, H in (("min_lifetime", 2), ("nearest_urgent", 1), ("min_lifetime", 0)):
        cand = torch.as_tensor(rng.uniform(-0.5, 1.5, size=(4, K, 3)))                 # outside [0, 1] too
        valid = torch.as_tensor(rng.uniform(size=(4, K)) < 0.8)
        valid[0] = True
        got, _, n = check_lookahead(env, cand, valid, H, kind, make)
        inflight += n
        fin = got[np.isfinite(got).all(1)]
        unequal += sum(len(np.unique(r)) > 1 for r in fin)
        missing += int(np.isnan(got).all(1).sum())
    assert unequal >= 3
    if budget:
        assert missing >= 1 and inflight >= 3, (missing, inflight)


def test_branches_that_end_inside_the_horizon(host):
    scs = [_short_lived(), synthetic(40, 40, seed=3)]
    make = lambda R: BatchedWRSN(scs, num_agent=2, num_envs=R, device="cpu", warm_up_time=10)   # noqa: E731
    env = make(4)
    env.reset()
    cand = torch.as_tensor(np.random.default_rng(3).uniform(0.0, 1.0, size=(4, 2, 3)))
    _, ended, _ = check_lookahead(env, cand, torch.ones((4, 2), dtype=torch.bool), 40, "min_lifetime", make)
    assert ended >= 2


# ------------------------------------------------------------------ 4. the planner
def test_width_one_planner_is_the_rule(host):
    scs = [_short_lived(), synthetic(40, 40, seed=3)]
    for kind in KINDS:
        res, rec = [], []
        for ctl in (HeuristicController(kind), LookaheadController(kind, width=1, horizon=3)):
            env = BatchedWRSN(scs, num_agent=2, num_envs=4, scenario_index=[0, 1, 1, 0], device="cpu", warm_up_time=10)
            res.append({k: _np(v) for k, v in evaluate(env, ctl, episodes=2, max_decisions=12).items()})
            rec.append(_record(env))
        for n in res[0]:
            assert np.array_equal(res[0][n], res[1][n]), (kind, n)
        for x, y in zip(*rec):
            assert x.tobytes() == y.tobytes(), kind


def test_planner_picks_the_first_best_slot(host):
    env = _mixed(B=4)
    env.reset()
    ctl = LookaheadController("min_lifetime", width=4, horizon=2, charge_levels=(1.0, 0.2))
    action = torch.zeros((4, 3), dtype=torch.float64)
    not_zero = unequal = 0
    for t in range(12):
        cand, valid = ctl.candidates(env)
        assert cand.shape == (4, 12, 3)
        ctl.plan(env, action)
        values, best = (_np(x) for x in ctl.last)
        aid = _np(env.req.agent_id)
        c = _np(cand)
        for b in range(4):
            if aid[b] < 0:
                continue
            top = values[b].max()
            assert best[b] == np.flatnonzero(values[b] == top)[0] and values[b, best[b]] >= values[b, 0]
            assert np.array_equal(_bits(_np(action)[b]), _bits(c[b, best[b]]))
            not_zero += best[b] != 0
            unequal += len(np.unique(values[b][np.isfinite(values[b])])) > 1
        env.rollout_step(action)
    assert not_zero >= 3 and unequal >= 6


def test_rollout_takes_the_plan(host):
    env = _mixed(B=4)
    env.reset()
    ctl = LookaheadController("nearest_urgent", width=2, horizon=1, charge_levels=(1.0,))
    seen = []
    inner = env.rollout_step

    def spy(action, obs=None):
        rows = _np(env.req.agent_id) >= 0
        values, best = (_np(x) for x in ctl.last)
        cand, _ = ctl.candidates(env)
        want = _np(cand)[np.arange(4), best]
        assert np.array_equal(_bits(_np(action)[rows]), _bits(want[rows]))
        seen.append(int(rows.sum()))
        return inner(action, obs)

    env.rollout_step = spy
    try:
        obs, stats = rollout(env, ctl, 6)
    finally:
        del env.rollout_step
    assert len(seen) == 6 and sum(seen) > 0 and np.isfinite(stats["reward_sum"]) and obs.shape == (4, 4, 100, 100)


# ------------------------------------------------------------------ 5. GPU
@pytest.mark.gpu
def test_device_candidates_equal_the_host_build_on_a_gpu_snapshot(emu_built, tmp_path):
    helpers.use_cuda_build()
    B = 2304
    env = _mixed(B=B, device=GPU)
    obs = torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=GPU)
    act = torch.zeros((B, 3), dtype=torch.float64, device=GPU)
    env.reset()
    env.get_state(out=obs)
    for _ in range(12):
        env.linear_controller_action(obs, W_RANDOM, out=act)
        env.rollout_step(act, obs)
    env.raise_on_error()
    aids = [None] + [torch.full((B,), a, dtype=torch.int32, device=GPU) for a in range(env.M)]

    def run(e, dev):
        out = {}
        for kind in KINDS:
            for K in WIDTHS:
                for i, a in enumerate(aids):
                    a = None if a is None else a.to(dev)
                    x = torch.full((B, K, 3), SENTINEL, dtype=torch.float64, device=dev)
                    n = torch.full((B, K), NODE_SENTINEL, dtype=torch.int32, device=dev)
                    x, n = e.heuristic_candidates(kind, K, agent_id=a, out=x, node=n)
                    out[(kind, K, i)] = (_np(x), _np(n))
        return out

    dev = run(env, GPU)
    assert (_np(env.req.agent_id) >= 0).any()
    path = str(tmp_path / "rows.pt")
    env.snapshot().save(path)
    try:
        helpers.use_host_build()
        host = _mixed(B=B)
        host.restore(EnvSnapshot.load(path))
        for key, (x, n) in run(host, "cpu").items():
            assert np.array_equal(n, dev[key][1]), key
            assert np.array_equal(_bits(x), _bits(dev[key][0])), key
    finally:
        helpers.use_cuda_build_lazy()


@pytest.mark.gpu
@pytest.mark.parametrize("nodes,chargers", [(1000, 16), (1000, 3), (100, 16)])
def test_device_candidates_equal_the_host_build_and_the_restatement(emu_built, tmp_path, nodes, chargers):
    helpers.use_cuda_build()
    scs = [synthetic(nodes, nodes, seed=s) for s in (11, 12)]
    B = 64
    env = BatchedWRSN(scs, num_agent=chargers, num_envs=B, device=GPU, step_budget=100)
    acts = np.random.default_rng(nodes + chargers).uniform(0.0, 1.0, size=(30, B, 3))
    acts[..., 2] *= 0.05
    env.reset()
    for t in range(30):
        env.rollout_step(torch.as_tensor(acts[t], device=GPU))
    env.raise_on_error()
    counts = check_all(env, widths=(1, 8, 32))
    assert (counts >= 32).sum() >= B
    dev = {(kind, K): tuple(_np(x) for x in env.heuristic_candidates(kind, K)) for kind in KINDS for K in (8, 32)}
    path = str(tmp_path / "rows.pt")
    env.snapshot().save(path)
    try:
        helpers.use_host_build()
        host = BatchedWRSN(scs, num_agent=chargers, num_envs=B, device="cpu", step_budget=100)
        host.restore(EnvSnapshot.load(path))
        for (kind, K), (x, n) in dev.items():
            hx, hn = (_np(t) for t in host.heuristic_candidates(kind, K))
            rows = _np(host.req.agent_id) >= 0
            assert np.array_equal(hn[rows], n[rows]) and np.array_equal(_bits(hx[rows]), _bits(x[rows])), (kind, K)
    finally:
        helpers.use_cuda_build_lazy()


@pytest.mark.gpu
@pytest.mark.parametrize("budget", [0, 60])
def test_device_lookahead_equals_replays(budget):
    helpers.use_cuda_build()
    env = _mixed(B=16, device=GPU, step_budget=budget)
    make = lambda R: _mixed(B=R, device=GPU, step_budget=budget)   # noqa: E731
    env.reset()
    rng = np.random.default_rng(20 + budget)
    for t in range(10):
        env.rollout_step(torch.as_tensor(rng.uniform(0.0, 1.0, size=(16, 3)) * [1.0, 1.0, 0.1], device=GPU))
    cand, _ = env.heuristic_candidates("min_lifetime", 4)
    cand = cand + torch.as_tensor(rng.uniform(-0.3, 0.3, size=(16, 4, 3)), device=GPU)
    valid = torch.as_tensor(rng.uniform(size=(16, 4)) < 0.85, device=GPU)
    got, _, inflight = check_lookahead(env, cand.contiguous(), valid, 3, "nearest_urgent", make)
    assert inflight >= 1 or not budget
    assert sum(len(np.unique(r)) > 1 for r in got[np.isfinite(got).all(1)]) >= 3


@pytest.mark.gpu
def test_planner_on_the_headline_workload():
    helpers.use_cuda_build()
    scs = [synthetic(100, 100, seed=1000 + k) for k in range(4)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=4096, device=GPU, step_budget=100)
    env.reset()
    ctl = LookaheadController("min_lifetime", width=8, horizon=4, charge_levels=(1.0,))
    out = torch.zeros((4096, 3), dtype=torch.float64, device=GPU)
    ctl.plan(env, out)                                                # every row holds its first request
    values, best = ctl.last
    decided = env.req.agent_id >= 0
    assert int(decided.sum()) > 0 and bool(torch.isnan(values[~decided]).all())
    assert bool(torch.isfinite(values[decided, 0]).all()) and int((best[decided] != 0).sum()) > 0
    obs, stats = rollout(env, ctl, 4)                                 # long charges: most rows are in flight afterwards
    assert stats["decisions"] > 0 and np.isfinite(stats["reward_sum"]) and bool(torch.isfinite(obs).all())
