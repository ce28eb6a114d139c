"""Rule rollouts on the device (BatchedWRSN.rule_rollout, wrsn_rule_rollout): the rule decides inside the step kernel and the row
keeps stepping.  Checked byte for byte against ``restate`` below, the same accounting driven from the host one request at a time
(heuristic_action + step(mask=running), with batched.episode_ends / episode_step), on the host build of the kernel source and
(``-m gpu``) on the device, which must also equal the host build.  Each regime a case is meant to reach is counted, and the case
fails below a floor.  The device and the host build differ only where update_reward's reciprocals let them (DESIGN §4.1):
rewards, returns and the chargers' exclusive rewards are compared to 1e-9 there, everything else bit for bit."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, EnvSnapshot, HeuristicController, LookaheadController, _lib, evaluate, synthetic
from multi_agent_rl_wrsn_b200.batched import episode_ends, episode_step
from tests import helpers
from tests import parity_cases as pc
from tests import test_lookahead as tl
from tests.helpers import REPO

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
KINDS = ("min_lifetime", "nearest_urgent")


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


# ------------------------------------------------------------------ the host-driven restatement
def restate(env, kind, limit, first_action=None, running=None):
    """rule_rollout's result, one request at a time from the host: at every request the rows that end their episode leave
    (episode_ends), the others get the rule's action (first_action for a row's first decision) and one step(mask=running)
    (episode_step).  -> (returns, decisions, -2 requests stepped)."""
    B, dev = env.B, env.device
    run = (env.req.agent_id >= 0) if running is None else running.clone()
    dec = torch.zeros(B, dtype=torch.int64, device=dev)
    ret = torch.zeros(B, dtype=torch.float64, device=dev)
    action = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    implicit = 0
    while True:
        _, ended = episode_ends(env.req, run, dec, limit)
        run &= ~ended
        if not bool(run.any()):
            break
        env.heuristic_action(kind, out=action)
        if first_action is not None:
            action = torch.where((dec == 0)[:, None], first_action, action)
        implicit += int((run & (env.req.agent_id == -2)).sum())
        episode_step(env, run, action, dec, ret)
    env.raise_on_error()
    return ret, dec, implicit


def record(env, budget):
    """The state records without the engine's scratch field and the request record.  With a step budget the records leave out
    hdr NRESUME / NBATCH, the times of the grid processes that have stopped (NET_T, UR_T, UNTIL_T where NET_ON, UR_ON, UNTIL_ON
    are 0: the last value the clock stored, not state) and stats[:, 1]: a launch-wide budget cuts steps at other places than a
    budget per step, which only changes those and the order in which the simulated seconds of a step are summed."""
    end = int(env._foff[env.E["WRSN_F_SCRATCH"]])
    st = _np(env.state[:, :end])
    q = env.req
    stats = _np(q.stats)
    if budget:
        hdr0 = int(env._foff[env.E["WRSN_F_HDR"]])
        col = lambda f: hdr0 + 8 * env.E["WRSN_H_" + f]          # noqa: E731
        for f in ("NRESUME", "NBATCH"):
            st[:, col(f):col(f) + 8] = 0
        for f in ("NET", "UR", "UNTIL"):
            off = st[:, col(f + "_ON"):col(f + "_ON") + 8].copy().view(np.float64)[:, 0] == 0.0
            st[off, col(f + "_T"):col(f + "_T") + 8] = 0
        stats[:, 1] = 0.0
    return [st, stats] + [_np(getattr(q, f)) for f in ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "sticky")]


class Spy:
    """Counts, per launch of wrsn_rule_rollout, the rows left in flight and the rows stopped by launch_max."""

    def __init__(self, env, limit, decisions):
        self.env, self.limit, self.dec = env, limit, decisions
        self.inflight = self.capped = self.launches = 0
        self.inner = env._call

    def __call__(self, fn, *args):
        self.inner(fn, *args)
        if getattr(fn, "__name__", "") == "wrsn_rule_rollout":
            aid = _np(self.env.req.agent_id)
            run = np.frombuffer(ctypes.string_at(args[4], self.env.B) if self.env.device.type == "cpu" else b"", np.uint8)
            self.launches += 1
            self.inflight += int((aid == -4).sum())
            if run.size:
                self.capped += int(((run != 0) & (aid >= 0) & (_np(self.dec) < self.limit)).sum())


def check_rollout(a, b, kind, limit, first=None, running=None, launch_max=None, budget=0):
    """a.rule_rollout against restate on b (the same rows): returns, decisions, running, state and request records, byte for
    byte.  -> regime counts."""
    dec = torch.zeros(a.B, dtype=torch.int64, device=a.device)
    spy = Spy(a, limit, dec)
    a._call = spy
    try:
        ret, dec, run = a.rule_rollout(kind, limit, first_action=first, running=running, decisions=dec, launch_max=launch_max)
    finally:
        del a._call
    want_ret, want_dec, implicit = restate(b, kind, limit, first, running)
    assert not bool(run.any())
    assert np.array_equal(_np(dec), _np(want_dec)), (kind, limit, _np(dec), _np(want_dec))
    assert np.array_equal(_bits(_np(ret)), _bits(_np(want_ret))), (kind, limit, _np(ret), _np(want_ret))
    for i, (x, y) in enumerate(zip(record(a, budget), record(b, budget))):
        assert x.tobytes() == y.tobytes(), (kind, limit, i, np.nonzero((x != y).reshape(len(x), -1).any(1))[0])
    aid = _np(a.req.agent_id)
    d = _np(dec)
    return dict(terminal=int((aid == -1).sum()), limited=int(((aid != -1) & (d >= limit)).sum()), implicit=implicit,
                inflight=spy.inflight, capped=spy.capped)


def _pair(make, prepare):
    a = make()
    prepare(a)
    snap = a.snapshot()
    b = make()
    b.restore(snap)
    return a, b, snap


CASES = [("min_lifetime", 0, 1024, False), ("nearest_urgent", 1, 1, True), ("min_lifetime", 2, 3, True),
         ("nearest_urgent", 7, 3, False), ("min_lifetime", 7, 1, True), ("nearest_urgent", 40, 1024, True),
         ("min_lifetime", 40, 3, False)]


def _sweep(a, b, snap, budget, rng):
    tot = {}
    for kind, limit, lm, with_first in CASES:
        a.restore(snap)
        b.restore(snap)
        first = torch.as_tensor(rng.uniform(-0.5, 1.5, size=(a.B, 3)), device=a.device) if with_first else None
        running = None if limit == 0 else torch.ones(a.B, dtype=torch.bool, device=a.device)   # (None: the rows with a decider)
        for k, v in check_rollout(a, b, kind, limit, first=first, running=running, launch_max=lm, budget=budget).items():
            tot[k] = tot.get(k, 0) + v
    return tot


def _warm(budget):
    def prepare(env):
        env.reset()
        rng = np.random.default_rng(5 + budget)
        for t in range(6):
            env.rollout_step(torch.as_tensor(rng.uniform(0.0, 1.0, size=(env.B, 3)) * [1.0, 1.0, 0.3], device=env.device))
    return prepare


@pytest.mark.parametrize("budget,rounds", [(0, 0), (25, 0), (60, 2), (25, 2)])
def test_mixed_batch_equals_the_restatement(host, budget, rounds):
    make = lambda: tl._mixed(B=8, step_budget=budget, step_rounds=rounds)     # noqa: E731  82 / 98 / 132 / 100 nodes
    a, b, snap = _pair(make, _warm(budget))
    tot = _sweep(a, b, snap, budget, np.random.default_rng(budget + rounds))
    assert tot["limited"] >= 20 and tot["capped"] >= 10, tot
    if budget:
        assert tot["inflight"] >= 5, tot


def _short(budget=0):
    scs = [tl._short_lived(), synthetic(40, 40, seed=3)]
    return lambda: BatchedWRSN(scs, num_agent=2, num_envs=6, scenario_index=[0, 1, 0, 1, 0, 0], device="cpu",  # noqa: E731
                               warm_up_time=10, step_budget=budget)


@pytest.mark.parametrize("budget", [0, 25])
def test_short_lived_fields_end_inside_the_limit(host, budget):
    a, b, snap = _pair(_short(budget), lambda e: e.reset())
    tot = _sweep(a, b, snap, budget, np.random.default_rng(1 + budget))
    assert tot["terminal"] >= 10, tot


@pytest.mark.parametrize("budget", [0, 25])
def test_chargers_that_die_on_the_way(host, budget):
    """700 J chargers (the ep_deadmc_n50 fixture) die during the episode: implicit Nones (-2) are stepped inside a launch, and the
    rows end with every charger dead."""
    g = tl.golden("ep_deadmc_n50")
    make = lambda: BatchedWRSN(pc.sc_from_golden(g), num_agent=int(g["num_agent"]), mc_type=tl.mc_dict_of(g), num_envs=3,  # noqa: E731
                               device="cpu", step_budget=budget)
    a, b, snap = _pair(make, lambda e: e.reset())
    tot = {}
    for kind in KINDS:
        a.restore(snap)
        b.restore(snap)
        for k, v in check_rollout(a, b, kind, 400, running=torch.ones(3, dtype=torch.bool), launch_max=7, budget=budget).items():
            tot[k] = tot.get(k, 0) + v
        assert (_np(a.req.sticky) & 1).all()
    assert tot["implicit"] >= 2 and tot["terminal"] == 6, tot


def test_dead_chargers(host):
    """A dead charger (status 0) in some rows and every charger dead in others: the rows end on a request with flags bit 0."""
    def prepare(env):
        _warm(0)(env)
        mc = env.view("mc")
        mc[1, 0, env.E["WRSN_MC_STATUS"]] = 0.0
        mc[2, :, env.E["WRSN_MC_STATUS"]] = 0.0
        mc[5, :, env.E["WRSN_MC_STATUS"]] = 0.0
    a, b, snap = _pair(lambda: tl._mixed(B=8), prepare)
    tot = _sweep(a, b, snap, 0, np.random.default_rng(9))
    assert tot["terminal"] >= 2, tot
    a.restore(snap)
    a.rule_rollout("min_lifetime", 40, running=torch.ones(8, dtype=torch.bool))
    assert (_np(a.req.flags)[[2, 5]] & 1).all() and (_np(a.req.agent_id)[[2, 5]] == -1).all()


# ------------------------------------------------------------------ lookahead and evaluate through the rollout
@pytest.mark.parametrize("budget", [0, 60])
def test_deep_lookahead_equals_replays(host, budget):
    env = tl._mixed(B=4, step_budget=budget)
    make = lambda R: tl._mixed(B=R, step_budget=budget)               # noqa: E731
    env.reset()
    rng = np.random.default_rng(30 + budget)
    cand = torch.as_tensor(rng.uniform(-0.5, 1.5, size=(4, 2, 3)))
    got, _, _ = tl.check_lookahead(env, cand, torch.ones((4, 2), dtype=torch.bool), 50, "nearest_urgent", make)
    assert np.isfinite(got).all()


def test_lookahead_to_the_end_of_the_episode(host):
    scs = [tl._short_lived(), synthetic(40, 40, seed=3)]
    make = lambda R: BatchedWRSN(scs, num_agent=2, num_envs=R, scenario_index=np.arange(R) % 2 * 0, device="cpu",  # noqa: E731
                                 warm_up_time=10)
    env = make(4)
    env.reset()
    cand = torch.as_tensor(np.random.default_rng(4).uniform(0.0, 1.0, size=(4, 3, 3)))
    _, ended, _ = tl.check_lookahead(env, cand, torch.ones((4, 3), dtype=torch.bool), 400, "min_lifetime", make)
    assert ended == 12                                                # every branch reaches the episode's end


class _Wrapped:
    """The rule as a generic controller (make_action, no heuristic attribute): evaluate's per-request loop."""

    def __init__(self, kind):
        self.kind = kind

    def make_action(self, agent_id, state, info=None, wrsn=None):
        return self.env.heuristic_action(self.kind, agent_id=agent_id)


def _evaluate_both(make, kind, **kw):
    out = []
    for ctl in (HeuristicController(kind), _Wrapped(kind)):
        env = make()
        ctl.env = env
        res = {k: _np(v) for k, v in evaluate(env, ctl, **kw).items()}
        out.append((res, tl._record(env)))
    return out


def test_evaluate_equals_the_generic_loop(host):
    scs = [tl._short_lived(), synthetic(40, 40, seed=3)]
    make = lambda: BatchedWRSN(scs, num_agent=2, num_envs=4, scenario_index=[0, 1, 1, 0], device="cpu", warm_up_time=10)  # noqa: E731
    trunc = 0
    for kind in KINDS:
        (r0, rec0), (r1, rec1) = _evaluate_both(make, kind, episodes=2, max_decisions=25)
        for n in r0:
            assert r0[n].tobytes() == r1[n].tobytes(), (kind, n)
        for x, y in zip(rec0, rec1):
            assert x.tobytes() == y.tobytes(), kind
        trunc += int(r0["truncated"].sum())
        assert (~r0["truncated"]).sum() >= 2
    assert trunc >= 2


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
                  running=np.zeros(2, np.uint8), decisions=np.zeros(2, np.int64), returns=np.zeros(2, np.float64),
                  agent=np.full(2, -1, np.int32))

    def call(L, d, null=None, kind=0, limit=4, lm=16):
        p = {k: (None if k == null else a.ctypes.data) for k, a in arrays.items()}
        req = _lib.Request(p["agent"], None, None, None, None, None, None, None, None, None)
        rc = L.wrsn_rule_rollout(ctypes.byref(d), p["scen"], p["scen_id"], p["state"], p["running"], kind, None, limit, lm,
                                 p["decisions"], p["returns"], ctypes.byref(req), None)
        return rc, L.wrsn_last_error()

    mx = _lib.enums()["WRSN_ROLL_MAX"]
    cases = [(dict(finalize=False), {}, b"dims not finalized"), ({}, dict(null="running"), b"NULL argument"),
             ({}, dict(null="decisions"), b"NULL argument"), ({}, dict(null="returns"), b"NULL argument"),
             ({}, dict(null="agent"), b"NULL argument"), ({}, dict(null="state"), b"NULL argument"),
             ({}, dict(kind=-1), b"heuristic kind -1"), ({}, dict(kind=2), b"heuristic kind 2"),
             ({}, dict(limit=-1), b"limit = -1 decisions"), ({}, dict(lm=0), b"launch_max = 0 decisions: 1 to %d" % mx),
             ({}, dict(lm=mx + 1), b"launch_max = %d" % (mx + 1))]
    for dkw, ckw, msg in cases:
        got = [call(L, dims(L, **dkw), **ckw) for L in libs]
        assert got[0] == got[1], (dkw, ckw, got)
        assert got[0][0] == -1 and msg in got[0][1], (dkw, ckw, got)
    for lm in (1, mx):                                                # the bounds are accepted (no row runs: nothing is read)
        assert call(libs[1], dims(libs[1]), lm=lm)[0] == 0


def test_python_refusals(host):
    env = tl._mixed(B=2, synth=False)
    env.reset()
    with pytest.raises(ValueError, match="kind"):
        env.rule_rollout("random", 3)
    with pytest.raises(ValueError, match="limit"):
        env.rule_rollout("min_lifetime", -1)
    for lm in (0, _lib.enums()["WRSN_ROLL_MAX"] + 1):
        with pytest.raises(ValueError, match="launch_max"):
            env.rule_rollout("min_lifetime", 3, launch_max=lm)
    with pytest.raises(ValueError, match="first_action"):
        env.rule_rollout("min_lifetime", 3, first_action=torch.zeros((2, 3), dtype=torch.float32))
    with pytest.raises(ValueError, match="decisions"):
        env.rule_rollout("min_lifetime", 3, decisions=torch.zeros(2, dtype=torch.int32))
    with pytest.raises(ValueError, match="returns"):
        env.rule_rollout("min_lifetime", 3, returns=torch.zeros(3, dtype=torch.float64))
    with pytest.raises(ValueError, match="running"):
        env.rule_rollout("min_lifetime", 3, running=torch.ones(3, dtype=torch.bool))


# ------------------------------------------------------------------ GPU
def _exact_and_close(env):
    """The records split into what the device and the host build must give bit for bit and what update_reward's reciprocals
    let differ in the last bits (DESIGN §4.1): the rewards, detail and the chargers' exclusive reward (mc EXCL)."""
    end = int(env._foff[env.E["WRSN_F_SCRATCH"]])
    st = _np(env.state[:, :end])
    mc0 = int(env._foff[env.E["WRSN_F_MC"]])
    excl = []
    for j in range(env.M):
        o = mc0 + 8 * (j * env.E["WRSN_MC_LEN"] + env.E["WRSN_MC_EXCL"])
        excl.append(st[:, o:o + 8].copy().view(np.float64)[:, 0])
        st[:, o:o + 8] = 0
    q = env.req
    exact = [st] + [_np(getattr(q, f)) for f in ("agent_id", "terminal", "now", "action", "flags", "sticky", "stats")]
    return exact, [np.stack(excl, 1), _np(q.reward), _np(q.detail)]


def _device_vs_host(make_dev, make_host, prepare, kinds_limits, tmp_path, budget):
    """rule_rollout on the device against the host build on the same rows (a snapshot): decisions and records bit for bit,
    returns, rewards and the exclusive rewards to 1e-9 (as the engine's own device / host comparison); and the device against
    restate on the device, byte for byte."""
    helpers.use_cuda_build()
    env = make_dev()
    prepare(env)
    path = str(tmp_path / "rows.pt")
    env.snapshot().save(path)
    snap = env.snapshot()
    dev = []
    for kind, limit, lm in kinds_limits:
        env.restore(snap)
        first = torch.full((env.B, 3), 0.5, dtype=torch.float64, device=env.device)
        ret, dec, _ = env.rule_rollout(kind, limit, first_action=first, launch_max=lm)
        dev.append((_np(ret), _np(dec), _exact_and_close(env)))
    twin = make_dev()
    env.restore(snap)
    twin.restore(snap)
    kind, limit, lm = kinds_limits[0]
    check_rollout(env, twin, kind, limit, launch_max=lm, budget=budget)
    try:
        helpers.use_host_build()
        h = make_host()
        hs = EnvSnapshot.load(path)
        for (kind, limit, lm), (ret, dec, rec) in zip(kinds_limits, dev):
            h.restore(hs)
            first = torch.full((h.B, 3), 0.5, dtype=torch.float64)
            hr, hd, _ = h.rule_rollout(kind, limit, first_action=first, launch_max=lm)
            assert np.array_equal(_np(hd), dec), (kind, limit)
            np.testing.assert_allclose(_np(hr), ret, rtol=1e-9, atol=1e-12)
            exact, close = _exact_and_close(h)
            for x, y in zip(exact, rec[0]):
                assert x.tobytes() == y.tobytes(), (kind, limit)
            for x, y in zip(close, rec[1]):
                np.testing.assert_allclose(x, y, rtol=1e-9, atol=1e-12, equal_nan=True)
    finally:
        helpers.use_cuda_build_lazy()
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("budget", [0, 100])
def test_device_equals_the_host_build_on_a_headline_snapshot(emu_built, tmp_path, budget):
    B = 2304
    make = lambda dev: (lambda: tl._mixed(B=B, device=dev, step_budget=budget))   # noqa: E731

    def prepare(env):
        env.reset()
        obs = torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=env.device)
        act = torch.zeros((B, 3), dtype=torch.float64, device=env.device)
        env.get_state(out=obs)
        for _ in range(8):
            env.linear_controller_action(obs, tl.W_RANDOM, out=act)
            env.rollout_step(act, obs)
        env.raise_on_error()
    _device_vs_host(make(GPU), make("cpu"), prepare, [("min_lifetime", 5, 1024), ("nearest_urgent", 12, 3)], tmp_path, budget)


@pytest.mark.gpu
@pytest.mark.parametrize("nodes,chargers", [(1000, 16), (1000, 3), (128, 3), (129, 3)])
def test_device_group_builds_equal_the_host_build(emu_built, tmp_path, nodes, chargers):
    """1000 nodes run the multi-warp build on 128 threads (the cross-warp reduction), 128 nodes the one-warp build, 129 two warps."""
    scs = [synthetic(nodes, nodes, seed=s) for s in (11, 12)]
    B = 48
    make = lambda dev: (lambda: BatchedWRSN(scs, num_agent=chargers, num_envs=B, device=dev, step_budget=100))   # noqa: E731

    def prepare(env):
        env.reset()
        acts = np.random.default_rng(nodes + chargers).uniform(0.0, 1.0, size=(6, B, 3)) * [1.0, 1.0, 0.05]
        for t in range(6):
            env.rollout_step(torch.as_tensor(acts[t], device=env.device))
    helpers.use_cuda_build()
    assert int(make(GPU)().dims.threads) == (128 if nodes == 1000 else (32 if nodes == 128 else 64))
    _device_vs_host(make(GPU), make("cpu"), prepare, [("nearest_urgent", 6, 1024), ("min_lifetime", 4, 1)], tmp_path, 100)


@pytest.mark.gpu
def test_device_evaluate_equals_the_host_build(emu_built):
    scs = [tl._short_lived(), synthetic(60, 60, seed=3)]
    res = []
    for dev in (GPU, "cpu"):
        (helpers.use_cuda_build if dev == GPU else helpers.use_host_build)()
        try:
            env = BatchedWRSN(scs, num_agent=2, num_envs=16, device=dev, warm_up_time=10)
            res.append({k: _np(v) for k, v in evaluate(env, HeuristicController("nearest_urgent"), episodes=2, max_decisions=30).items()})
        finally:
            helpers.use_cuda_build_lazy()
    for n in ("lifetime", "decisions", "truncated"):
        assert res[0][n].tobytes() == res[1][n].tobytes(), n
    np.testing.assert_allclose(res[0]["return"], res[1]["return"], rtol=1e-9, atol=1e-12)   # update_reward's reciprocals


@pytest.mark.gpu
def test_device_planner_on_the_headline_workload():
    helpers.use_cuda_build()
    scs = [synthetic(100, 100, seed=1000 + k) for k in range(4)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=4096, device=GPU, step_budget=100)
    env.reset()
    ctl = LookaheadController("min_lifetime", width=8, horizon=16)
    out = torch.zeros((4096, 3), dtype=torch.float64, device=GPU)
    ctl.plan(env, out)
    values, best = ctl.last
    decided = env.req.agent_id >= 0
    assert int(decided.sum()) > 0 and bool(torch.isfinite(values[decided, 0]).all())
