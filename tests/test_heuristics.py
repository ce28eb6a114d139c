"""Hand-written charging rules (BatchedWRSN.heuristic_action, wrsn_heuristic_action), HeuristicController and controllers.evaluate.

The rule is checked bit for bit against oracle/heuristic_oracle.py, a numpy restatement over the state views, on the host build of
the kernel source and (``-m gpu``) on k_heuristic; the device must also equal the host build byte for byte on the same rows."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, EnvSnapshot, HeuristicController, _lib, evaluate, rollout, synthetic
from oracle import heuristic_oracle as ho
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO, golden, mc_dict_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
GOLDEN3 = ("ep_basic_n50", "ep_full_n100", "ep_full_n200")      # 82 / 98 / 132 nodes
W_RANDOM = (1.0, 1.0, -10.0, 1.0)
KINDS = ho.KINDS
SENTINEL = 7.25


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


def _mixed(B=8, device="cpu", synth=True, **kw):
    gs = [golden(n) for n in GOLDEN3]
    scs = [pc.sc_from_golden(g) for g in gs] + ([synthetic(100, 100, seed=1000)] if synth else [])
    return BatchedWRSN(scs, num_agent=kw.pop("num_agent", 3), mc_type=mc_dict_of(gs[0]), num_envs=B, device=device, **kw)


def _rows(env):
    """Host copies of what the rule reads, per row."""
    E = env.E
    energy, cs, status, mc = _np(env.view("energy")), _np(env.view("cs")), _np(env.view("status")), _np(env.view("mc"))
    sid = _np(env.scen_id)
    for b in range(env.B):
        st = env.statics[int(sid[b])]
        m = mc[b, :env.M]
        yield b, dict(n=st["N"], x=np.asarray(st["x"], np.float64), y=np.asarray(st["y"], np.float64), energy=energy[b], cs=cs[b],
                      status=status[b], mc_x=m[:, E["WRSN_MC_X"]], mc_y=m[:, E["WRSN_MC_Y"]], mc_status=m[:, E["WRSN_MC_STATUS"]],
                      mc_dest_x=m[:, E["WRSN_MC_CPA0"]], mc_dest_y=m[:, E["WRSN_MC_CPA1"]], par=st["par"])


def oracle(env, kind, agent_id=None):
    """The restatement's actions [B, 3] and chosen nodes [B] (rows without a deciding charger: NaN / -2)."""
    aid = _np(env.req.agent_id if agent_id is None else torch.as_tensor(agent_id))
    out, pick = np.full((env.B, 3), np.nan), np.full(env.B, -2)
    for b, r in _rows(env):
        a = int(aid[b])
        if a < 0 or a >= env.M:
            continue
        pick[b] = ho.choose(kind, a, r["n"], r["x"], r["y"], r["energy"], r["cs"], r["status"], r["mc_x"], r["mc_y"], r["mc_status"],
                            r["mc_dest_x"], r["mc_dest_y"], r["par"])
        out[b] = ho.action(pick[b], a, r["x"], r["y"], r["energy"], r["mc_x"], r["mc_y"], r["par"])
    return out, pick


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.int64)


def check_equal(env, kind, agent_id=None):
    """heuristic_action == the restatement, bit for bit; rows without a deciding charger keep the sentinel."""
    out = torch.full((env.B, 3), SENTINEL, dtype=torch.float64, device=env.device)
    got = _np(env.heuristic_action(kind, agent_id=agent_id, out=out))
    want, pick = oracle(env, kind, agent_id)
    skip = pick == -2
    want[skip] = SENTINEL
    assert np.array_equal(_bits(got), _bits(want)), (kind, np.nonzero((_bits(got) != _bits(want)).any(1))[0][:8])
    return pick


# ------------------------------------------------------------------ 1. host build == restatement
def test_mixed_batch_equals_the_restatement(host):
    env = _mixed(B=8)
    env.reset()
    for kind in KINDS:
        check_equal(env, kind)
        for a in range(env.M):                       # every charger as the decider: other chargers' claims differ
            check_equal(env, kind, torch.full((env.B,), a, dtype=torch.int32))
    acts = np.random.default_rng(4).uniform(0.0, 1.0, size=(40, env.B, 3))
    acts[..., 2] *= 0.1
    for t in range(40):
        env.rollout_step(torch.as_tensor(acts[t]))
    assert (_np(env.req.stats)[:, 0] >= 40).all()
    picks = []
    for kind in KINDS:
        picks.append(check_equal(env, kind))
        for a in range(env.M):
            check_equal(env, kind, torch.full((env.B,), a, dtype=torch.int32))
    assert (picks[0] >= 0).any()


# ------------------------------------------------------------------ 2. edited states
def _edit_env(B=2):
    env = _mixed(B=B, synth=False)
    env.reset()
    return env


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


def _pick(env, kind, b=0, a=0):
    aid = torch.full((env.B,), a, dtype=torch.int32)
    return int(check_equal(env, kind, aid)[b])


def _lifetime_floor(env, b, nodes, life):
    """Give `nodes` the lifetime `life` (cs = 1), every other alive node of row b a longer one."""
    thr = env.statics[int(env.scen_id[b])]["par"]["THR"]
    e, cs = env.view("energy"), env.view("cs")
    n = int(env.num_nodes[b])
    cs[b, :n] = 1.0
    e[b, :n] = thr + 1e6
    for i in nodes:
        e[b, i] = thr + life


def test_equal_lifetimes_go_to_the_lowest_id(host):
    env = _edit_env()
    _clear_claims(env, 0)
    par = env.statics[0]["par"]
    _lifetime_floor(env, 0, (31, 9, 20), 2.0 * (par["MTM"] + par["CTM"]))    # the lowest, but not urgent
    for kind in KINDS:
        assert _pick(env, kind) == 9


def test_node_without_traffic_is_never_chosen_over_another(host):
    env = _edit_env()
    _clear_claims(env, 0)
    _lifetime_floor(env, 0, (4,), 50.0)
    env.view("energy")[0, 2] = env.statics[0]["par"]["THR"] + 1e-3   # the lowest energy, but no traffic
    env.view("cs")[0, 2] = 0.0
    for kind in KINDS:
        assert _pick(env, kind) == 4
    st = env.view("status")
    st[0, :] = 0
    st[0, 2] = 1                                                      # the only alive node: chosen after all
    for kind in KINDS:
        assert _pick(env, kind) == 2


def test_every_alive_node_claimed_falls_back_to_all_alive(host):
    env = _edit_env()
    _clear_claims(env, 0)
    st = env.view("status")
    st[0, :] = 0
    st[0, 7] = st[0, 12] = 1
    _lifetime_floor(env, 0, (12,), 30.0)
    x7, y7 = _xy(env, 0, 7)
    x12, y12 = _xy(env, 0, 12)
    _set_mc(env, 0, 1, STATUS=1.0, CPA0=x7, CPA1=y7)
    _set_mc(env, 0, 2, STATUS=1.0, CPA0=x12, CPA1=y12)
    for kind in KINDS:
        assert _pick(env, kind, a=0) == 12
    _set_mc(env, 0, 2, CPA0=-1e6, CPA1=-1e6)                          # node 12 free again: node 7 stays claimed
    for kind in KINDS:
        assert _pick(env, kind, a=0) == 12
    _set_mc(env, 0, 1, CPA0=x12, CPA1=y12)                            # now 12 is claimed and 7 is the only candidate
    for kind in KINDS:
        assert _pick(env, kind, a=0) == 7


def test_a_dead_charger_claims_nothing(host):
    env = _edit_env()
    _clear_claims(env, 0)
    _lifetime_floor(env, 0, (15,), 20.0)
    x, y = _xy(env, 0, 15)
    _set_mc(env, 0, 1, STATUS=0.0, CPA0=x, CPA1=y)
    assert _pick(env, "min_lifetime", a=0) == 15
    _set_mc(env, 0, 1, STATUS=1.0)
    assert _pick(env, "min_lifetime", a=0) != 15
    assert _pick(env, "min_lifetime", a=1) == 15                      # its own destination does not claim for itself


def test_padding_nodes_are_never_chosen(host):
    env = _mixed(B=3, synth=False)                                    # rows 82 / 98 / 132 nodes, N = 132
    env.reset()
    _clear_claims(env, 0)
    n0 = int(env.num_nodes[0])
    assert n0 == 82 and env.N == 132
    thr = env.statics[0]["par"]["THR"]
    env.view("status")[0, n0:] = 1
    env.view("energy")[0, n0:] = thr + 1e-6
    env.view("cs")[0, n0:] = 1.0
    for kind in KINDS:
        assert 0 <= _pick(env, kind) < n0


def test_nearest_urgent(host):
    env = _edit_env()
    _clear_claims(env, 0)
    par = env.statics[0]["par"]
    horizon = par["MTM"] + par["CTM"]
    _lifetime_floor(env, 0, (), 0.0)
    env.view("energy")[0, :int(env.num_nodes[0])] = par["THR"] + 2.0 * horizon   # nobody urgent
    env.view("energy")[0, 40] = par["THR"] + 1.5 * horizon
    assert _pick(env, "nearest_urgent") == _pick(env, "min_lifetime") == 40
    # two urgent nodes: the nearer one has the longer lifetime
    xa, ya = _xy(env, 0, 3)
    _set_mc(env, 0, 0, X=xa, Y=ya)
    far = int(np.argmax([np.hypot(_xy(env, 0, i)[0] - xa, _xy(env, 0, i)[1] - ya) for i in range(int(env.num_nodes[0]))]))
    env.view("energy")[0, 3] = par["THR"] + 0.9 * horizon
    env.view("energy")[0, far] = par["THR"] + 0.1 * horizon
    assert _pick(env, "nearest_urgent") == 3
    assert _pick(env, "min_lifetime") == far


def test_charge_fraction_limits(host):
    env = _edit_env()
    _clear_claims(env, 0)
    par = env.statics[0]["par"]
    st = env.view("status")
    st[0, :] = 0
    st[0, 11] = 1
    aid = torch.zeros(env.B, dtype=torch.int32)
    env.view("energy")[0, 11] = par["CAP"]
    assert float(env.heuristic_action("min_lifetime", agent_id=aid)[0, 2]) == 0.0
    env.view("energy")[0, 11] = np.nextafter(par["THR"], np.inf)
    assert float(env.heuristic_action("min_lifetime", agent_id=aid)[0, 2]) == 1.0
    for kind in KINDS:
        assert _pick(env, kind) == 11
    st[0, 11] = 0                                                    # no alive node: stay, charge 0
    _set_mc(env, 0, 0, X=par["F0"], Y=par["F3"])
    got = _np(env.heuristic_action("nearest_urgent", agent_id=aid))[0]
    assert got.tolist() == [0.0, 1.0, 0.0]
    assert _pick(env, "min_lifetime") == -1


def test_rows_without_a_decider_are_untouched(host):
    env = _mixed(B=6, synth=False)
    env.reset()
    aid = torch.tensor([-1, 0, -4, 2, -2, 1], dtype=torch.int32)
    for kind in KINDS:
        out = torch.full((6, 3), SENTINEL, dtype=torch.float64)
        got = _np(env.heuristic_action(kind, agent_id=aid, out=out))
        assert (got[[0, 2, 4]] == SENTINEL).all() and not (got[[1, 3, 5]] == SENTINEL).any()
        check_equal(env, kind, aid)


# ------------------------------------------------------------------ 3. the controller and the evaluator
def test_heuristic_controller_rollout_hands_the_rule_to_step(host):
    env = _mixed(B=4)
    env.reset()
    for kind in KINDS:
        seen = []
        inner = env.rollout_step

        def spy(action, obs=None):
            want, pick = oracle(env, kind)
            rows = pick != -2
            assert np.array_equal(_bits(_np(action)[rows]), _bits(want[rows]))
            seen.append(int(rows.sum()))
            return inner(action, obs)

        env.rollout_step = spy
        try:
            _, stats = rollout(env, HeuristicController(kind), 100)
        finally:
            del env.rollout_step
        assert len(seen) == 100 and sum(seen) > 0 and np.isfinite(stats["reward_sum"])


def test_single_environment_facade(host):
    from multi_agent_rl_wrsn_b200 import WRSN
    w = WRSN(synthetic(50, 50, seed=2), None, 3, density_map=False)
    r = w.reset()
    for kind in KINDS:
        a = r["agent_id"]
        x = HeuristicController(kind).make_action(a, r["state"], r["info"], wrsn=w)
        want = _np(w._b.heuristic_action(kind, agent_id=torch.tensor([a], dtype=torch.int32)))[0]
        assert x.shape == (3,) and np.array_equal(_bits(x), _bits(want))
        r = w.step(a, x)
        assert r is not None and r["agent_id"] is not None


def _short_lived():
    """A small network whose nodes start barely above threshold: it dies after a few decisions."""
    from multi_agent_rl_wrsn_b200.scenario import DEFAULT_NODE_PHY
    spe = dict(DEFAULT_NODE_PHY)
    spe["capacity"] = spe["threshold"] * 1.05
    return synthetic(30, 30, seed=7, node_phy_spe=spe)


def _manual_episodes(sc, kind, episodes, cap, warm_up):
    """One row alone, driven by hand: reset, step with the rule until the network is dead or `cap` decisions are made."""
    env = BatchedWRSN([sc], num_agent=2, num_envs=1, device="cpu", warm_up_time=warm_up)
    out = []
    for _ in range(episodes):
        req = env.reset()
        dec, ret = 0, 0.0
        while True:
            a = int(req.agent_id[0])
            if a == -1:
                out.append((float(req.now[0]) - warm_up, ret, dec, False))
                break
            if a != -4 and dec >= cap:
                out.append((float(req.now[0]) - warm_up, ret, dec, True))
                break
            act = env.heuristic_action(kind)
            req = env.step(torch.tensor([max(a, -1)], dtype=torch.int32), act)
            dec += a >= 0
            r = float(req.reward[0])
            ret += 0.0 if r != r else r
    return out


def test_evaluate_matches_a_manual_loop(host):
    scs = [_short_lived(), synthetic(40, 40, seed=3)]
    cap, E, warm = 6, 2, 10
    env = BatchedWRSN(scs, num_agent=2, num_envs=4, scenario_index=[0, 1, 1, 0], device="cpu", warm_up_time=warm)
    for kind in KINDS:
        res = evaluate(env, HeuristicController(kind), episodes=E, max_decisions=cap)
        assert set(res) == {"lifetime", "return", "decisions", "truncated"}
        assert all(v.shape == (4, E) for v in res.values())
        want = {k: _manual_episodes(scs[k], kind, E, cap, warm) for k in (0, 1)}
        for b, k in enumerate((0, 1, 1, 0)):
            for e in range(E):
                life, ret, dec, trunc = want[k][e]
                assert float(res["lifetime"][b, e]) == life, (kind, b, e)
                assert float(res["return"][b, e]) == ret, (kind, b, e)
                assert int(res["decisions"][b, e]) == dec and bool(res["truncated"][b, e]) == trunc, (kind, b, e)
        assert not res["truncated"][[0, 3]].any() and res["truncated"][[1, 2]].all()   # one network dies, the other is cut
        assert (res["decisions"][[1, 2]] == cap).all() and (res["decisions"][[0, 3]] < cap).all()


# ------------------------------------------------------------------ 4. refusals
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
                  agent=np.full(2, -1, np.int32), action=np.zeros(6, np.float64))

    def call(L, d, null=None, kind=0):
        p = {k: (None if k == null else a.ctypes.data) for k, a in arrays.items()}
        rc = L.wrsn_heuristic_action(ctypes.byref(d), p["scen"], p["scen_id"], p["state"], p["agent"], kind, p["action"], None)
        return rc, L.wrsn_last_error()

    cases = [(dict(finalize=False), {}, b"dims not finalized"), ({}, dict(null="action"), b"NULL argument"),
             ({}, dict(null="agent"), b"NULL argument"), ({}, dict(kind=-1), b"heuristic kind -1"),
             ({}, dict(kind=2), b"heuristic kind 2")]
    for dkw, ckw, msg in cases:
        got = [call(L, dims(L, **dkw), **ckw) for L in libs]
        assert got[0] == got[1], (dkw, ckw, got)
        assert got[0][0] == -1 and msg in got[0][1], (dkw, ckw, got)


def test_python_refusals(host):
    env = _mixed(B=2, synth=False)
    env.reset()
    with pytest.raises(ValueError, match="kind"):
        env.heuristic_action("farthest_first")
    with pytest.raises(ValueError, match="kind"):
        HeuristicController("random")
    for bad in (torch.zeros((2, 3), dtype=torch.float32), torch.zeros((3, 3), dtype=torch.float64),
                torch.zeros((3, 2), dtype=torch.float64).t()):
        with pytest.raises(ValueError, match="out"):
            env.heuristic_action("min_lifetime", out=bad)


# ------------------------------------------------------------------ 5. GPU
@pytest.mark.gpu
def test_device_equals_the_host_build_on_a_gpu_snapshot(emu_built, tmp_path):
    helpers.use_cuda_build()
    B = 2304
    env = _mixed(B=B, device=GPU)                                    # no step budget: every row ends the rollout holding a request
    obs = torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=GPU)
    act = torch.zeros((B, 3), dtype=torch.float64, device=GPU)
    env.reset()
    env.get_state(out=obs)
    for _ in range(12):
        env.linear_controller_action(obs, W_RANDOM, out=act)
        env.rollout_step(act, obs)
    env.raise_on_error()
    aids = [None] + [torch.full((B,), a, dtype=torch.int32, device=GPU) for a in range(env.M)]
    dev = {(k, i): _np(env.heuristic_action(k, agent_id=a, out=torch.full((B, 3), SENTINEL, dtype=torch.float64, device=GPU)))
           for k in KINDS for i, a in enumerate(aids)}
    assert (_np(env.req.agent_id) >= 0).any()
    path = str(tmp_path / "rows.pt")
    env.snapshot().save(path)
    try:
        helpers.use_host_build()
        host = _mixed(B=B)
        host.restore(EnvSnapshot.load(path))
        for (k, i), want in dev.items():
            a = None if aids[i] is None else aids[i].cpu()
            got = _np(host.heuristic_action(k, agent_id=a, out=torch.full((B, 3), SENTINEL, dtype=torch.float64)))
            assert np.array_equal(_bits(got), _bits(want)), (k, i)
    finally:
        helpers.use_cuda_build_lazy()


@pytest.mark.gpu
@pytest.mark.parametrize("nodes,chargers", [(1000, 3), (100, 16)])
def test_device_equals_the_restatement(nodes, chargers):
    helpers.use_cuda_build()
    scs = [synthetic(nodes, nodes, seed=s) for s in (11, 12)]
    B = 64
    env = BatchedWRSN(scs, num_agent=chargers, num_envs=B, device=GPU, step_budget=100)
    acts = np.random.default_rng(nodes + chargers).uniform(0.0, 1.0, size=(30, B, 3))
    acts[..., 2] *= 0.05
    env.reset()
    for kind in KINDS:
        check_equal(env, kind)
    for t in range(30):
        env.rollout_step(torch.as_tensor(acts[t], device=GPU))
    env.raise_on_error()
    for kind in KINDS:
        check_equal(env, kind)
        for a in range(chargers):
            check_equal(env, kind, torch.full((B,), a, dtype=torch.int32, device=GPU))


@pytest.mark.gpu
def test_heuristic_rollout_on_the_headline_workload():
    helpers.use_cuda_build()
    scs = [synthetic(100, 100, seed=1000 + k) for k in range(4)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=4096, device=GPU, step_budget=100)
    env.reset()
    for kind in KINDS:
        inner = env.rollout_step
        mism = torch.zeros((), dtype=torch.int64, device=GPU)

        def spy(action, obs=None):
            want = env.heuristic_action(kind)
            rows = env.req.agent_id >= 0
            mism.add_(((action != want).any(1) & rows).sum())
            return inner(action, obs)

        env.rollout_step = spy
        resets0 = float(env.req.stats[:, 2].sum())
        try:
            obs, stats = rollout(env, HeuristicController(kind), 64)
        finally:
            del env.rollout_step
        assert int(mism) == 0
        assert stats["decisions"] > 0 and np.isfinite(stats["reward_sum"])
        assert stats["episodes"] == float(env.req.stats[:, 2].sum()) - resets0
        assert not bool(((env.req.agent_id == -1) | (env.req.agent_id == -2)).any())   # finished episodes were reset
        assert obs.shape == (4096, 4, 100, 100) and bool(torch.isfinite(obs).all())


@pytest.mark.gpu
def test_evaluate_on_the_device_equals_the_host_build(emu_built):
    """Lifetimes, decisions and truncation exact; returns to 1e-9 (update_reward's reciprocals differ, DESIGN §4.1)."""
    results = {}
    for where in ("gpu", "cpu"):
        if where == "gpu":
            helpers.use_cuda_build()
        else:
            helpers.use_host_build()
        try:
            scs = [_short_lived(), synthetic(40, 40, seed=3), synthetic(100, 100, seed=1000)]
            env = BatchedWRSN(scs, num_agent=2, num_envs=8, device=GPU if where == "gpu" else "cpu", warm_up_time=10)
            results[where] = {k: {n: _np(v) for n, v in evaluate(env, HeuristicController(k), episodes=2, max_decisions=25).items()}
                              for k in KINDS}
        finally:
            if where == "cpu":
                helpers.use_cuda_build_lazy()
    for k in KINDS:
        g, h = results["gpu"][k], results["cpu"][k]
        for n in ("lifetime", "decisions", "truncated"):
            assert np.array_equal(g[n], h[n]), (k, n)
        np.testing.assert_allclose(g["return"], h["return"], rtol=1e-9, atol=1e-12)
