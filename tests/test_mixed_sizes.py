"""Batches whose scenarios have different node and target counts.

Every environment of a mixed batch must simulate exactly its own scenario: the reference's golden episodes row by row, the C
oracle row by row, and, byte for byte, what the same environment computes in a batch of its own scenario alone.  Each check
runs on the host emulation of the kernel source and (``-m gpu``) on the sm_100a kernels."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, _lib, synthetic
from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO, golden, mc_dict_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GOLDEN_MIXED = ("ep_basic_n50", "ep_edge_n50", "ep_longcharge_n50", "ep_full_n100", "ep_full_n200")   # 82 / 82 / 82 / 98 / 132 nodes
GPU = "cuda:0"
BACKENDS = ["cpu", pytest.param(GPU, marks=pytest.mark.gpu)]


@pytest.fixture(scope="module")
def emu_built():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)


@pytest.fixture(params=BACKENDS)
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


def _np(t):
    return t.detach().cpu().numpy().copy()


def _same(x, y):
    """Bit-for-bit equality (NaN rewards of rows without a request included)."""
    if x.shape != y.shape:
        return False
    if x.dtype == torch.float64:
        return torch.equal(x.contiguous().view(torch.int64), y.contiguous().view(torch.int64))
    if x.dtype == torch.float32:
        return torch.equal(x.contiguous().view(torch.int32), y.contiguous().view(torch.int32))
    return torch.equal(x, y)


def _golden_batch(names, device):
    gs = [golden(n) for n in names]
    for g in gs:
        assert int(g["num_agent"]) == 3 and int(g["map_size"]) == 100 and mc_dict_of(g) == mc_dict_of(gs[0])
    env = BatchedWRSN([pc.sc_from_golden(g) for g in gs], num_agent=3, mc_type=mc_dict_of(gs[0]), map_size=100,
                      scenario_index=np.arange(len(gs)), device=device)
    return gs, env


# ------------------------------------------------------------------ 1. golden episodes, one fixture per row
def _check_golden_mixed(names, device):
    gs, env = _golden_batch(names, device)
    B = len(gs)
    Ns, Ts = [int(v) for v in _np(env.num_nodes)], [int(v) for v in _np(env.num_targets)]
    assert env.N == max(Ns) and env.T == max(Ts)
    ns = [int(g["n"]) for g in gs]
    full = [{int(i): k for k, i in enumerate(g["full_state_idx"])} for g in gs]
    gpu = device != "cpu"
    for i in range(max(ns)):
        live = np.array([i < n for n in ns])
        if i == 0:
            req = env.reset()
        else:
            agent = np.array([int(g["fed_agent"][i]) if i < n else -1 for g, n in zip(gs, ns)], np.int32)
            action = np.stack([g["fed_action"][i] if i < n else np.zeros(3) for g, n in zip(gs, ns)])
            req = env.step(agent, action, mask=torch.as_tensor(live.astype(np.uint8)))
        aid, term, now, flags = _np(req.agent_id), _np(req.terminal), _np(req.now), _np(req.flags)
        status, level, tact = _np(env.view("status")), _np(env.view("level")), _np(env.targets_active())
        energy, cs, rr = _np(env.view("energy")), _np(env.view("cs")), _np(env.view("rr"))
        excl, action_out, reward = _np(env.mc("EXCL")), _np(req.action), _np(req.reward)
        for b in range(B):
            N, T = Ns[b], Ts[b]
            # padding columns keep their initial values throughout: dead, no energy, no level, no covered target
            assert not status[b, N:].any() and not energy[b, N:].any() and not cs[b, N:].any() and not rr[b, N:].any()
            assert (level[b, N:] == -1).all() and not tact[b, T:].any(), (b, i)
            if not live[b]:
                continue
            g, tag = gs[b], (names[b], i)
            assert int(aid[b]) == int(g["agent_id"][i]), tag
            assert int(term[b]) == int(g["terminal"][i]) and float(now[b]) == float(g["now"][i]) and int(flags[b]) == 0, tag
            assert np.array_equal(status[b, :N], g["status"][i]), tag
            assert np.array_equal(level[b, :N].astype(np.int32), g["level"][i]), tag
            assert np.array_equal(tact[b, :T], g["targets_active"][i]), tag
            np.testing.assert_allclose(energy[b, :N], g["energy"][i], rtol=pc.E_RTOL, err_msg=str(tag))
            np.testing.assert_allclose(cs[b, :N], g["cs"][i], rtol=pc.E_RTOL, err_msg=str(tag))
            np.testing.assert_allclose(excl[b], g["excl"][i], rtol=1e-9, atol=1e-15, err_msg=str(tag))
            if int(aid[b]) >= 0:
                assert np.array_equal(action_out[b], g["action"][i]), tag
                if i > 0:
                    np.testing.assert_allclose(float(reward[b]), float(g["reward"][i]), rtol=1e-9, atol=1e-18, err_msg=str(tag))
        want = [b for b in range(B) if live[b] and i in full[b]]
        if want:
            obs = _np(env.get_state(dtype=torch.float64))
            obs32 = _np(env.get_state(dtype=torch.float32)).astype(np.float64) if gpu else None
            for b in want:
                ref = gs[b]["full_state"][full[b][i]]
                np.testing.assert_allclose(obs[b], ref, rtol=1e-9, atol=1e-12, err_msg=str((names[b], i)))
                if gpu:
                    for ch in range(4):
                        tol = 1e-5 * max(float(np.abs(ref[ch]).max()), 1e-3)
                        assert float(np.abs(obs32[b][ch] - ref[ch]).max()) <= tol, (names[b], i, ch)
    fit, fmin = env.get_network_fitness()
    fit, fmin = _np(fit), _np(fmin)
    for b, g in enumerate(gs):
        assert not fit[b, Ts[b]:].any()
        if np.isfinite(g["fitness_min"][ns[b] - 1]):
            np.testing.assert_allclose(fmin[b], g["fitness_min"][ns[b] - 1], rtol=1e-12)
    assert float(_np(env.hdr("ERR")).max()) == 0.0
    return env


@pytest.mark.parametrize("rows", [5, 4])
def test_golden_episodes_mixed(dev, rows):
    """All five fixtures (largest 132 nodes: 64 threads per environment), and the first four (largest 98: one warp)."""
    env = _check_golden_mixed(GOLDEN_MIXED[:rows], dev)
    assert env.dims.threads == (64 if rows == 5 else 32)


# ------------------------------------------------------------------ 2. mixed batch == one batch per scenario, byte for byte
def _scenarios(kind):
    """"small": up to 128 nodes (one warp possible); "large": up to 150; "golden": the three golden sizes, whose narrow sources
    take the windowed float32 raster (the synthetic fields here are too small for it: their sources are wider)"""
    if kind == "golden":
        return [pc.sc_from_golden(golden(n)) for n in ("ep_basic_n50", "ep_full_n100", "ep_full_n200")]
    scs = [synthetic(num_nodes=40, num_targets=60, seed=41), pc.sc_from_golden(golden("ep_full_n100")),
           synthetic(num_nodes=128, num_targets=90, seed=42, num_gateways=4)]
    if kind == "large":
        scs += [synthetic(num_nodes=150, num_targets=170, seed=43, num_gateways=4), pc.sc_from_golden(golden("ep_full_n200"))]
    return scs


_VIEWS = ("energy", "rr", "cs", "esend", "logc", "nbef", "naft", "level", "parent", "status", "logtick", "ring")
_REQ = ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats", "sticky")


def _compare_rows(mixed, homo, rows, tag, obs):
    """Rows `rows` of the mixed batch against the whole homogeneous batch `homo`, field by field."""
    r = torch.as_tensor(rows, device=mixed.device)
    N, T = homo.N, homo.T
    for f in _REQ:
        assert _same(getattr(mixed.req, f)[r], getattr(homo.req, f)), (tag, f)
    for f in _VIEWS:
        assert _same(mixed.view(f)[r][..., :N], homo.view(f)), (tag, f)
    for f in ("hdr", "mc", "proc"):
        assert _same(mixed.view(f)[r], homo.view(f)), (tag, f)
    Tw, W = homo.dims.Tw, homo.dims.W
    assert _same(mixed.view("tact_words")[r][:, :Tw], homo.view("tact_words")) and not mixed.view("tact_words")[r][:, Tw:].any(), tag
    assert _same(mixed.view("conn_words")[r][..., :W], homo.view("conn_words")) and not mixed.view("conn_words")[r][..., W:].any(), tag
    assert _same(mixed.targets_active()[r][:, :T], homo.targets_active()), tag
    fm, fh = mixed.get_network_fitness(), homo.get_network_fitness()
    assert _same(fm[0][r][:, :T], fh[0]) and _same(fm[1][r], fh[1]), tag
    cm, ch = mixed.charge_rates(), homo.charge_rates()
    assert _same(cm[0][r][:, :N], ch[0]) and _same(cm[1][r], ch[1]), tag
    if obs:
        dtypes = (torch.float64,) if mixed.device.type == "cpu" else (torch.float64, torch.float32)
        for dt in dtypes:
            assert _same(mixed.get_state(dtype=dt)[r], homo.get_state(dtype=dt)), (tag, dt)


def _check_mixed_equals_homogeneous(device, scs, B, steps, threads, budget, rounds, controller=False, obs_every=4):
    sid = np.random.default_rng(7).permutation(np.arange(B) % len(scs))
    kw = dict(num_agent=3, device=device, threads=threads, step_budget=budget, step_rounds=rounds)
    mixed = BatchedWRSN(scs, num_envs=B, scenario_index=sid, **kw)
    rows = [np.nonzero(sid == s)[0] for s in range(len(scs))]
    homo = [BatchedWRSN([scs[s]], num_envs=len(rows[s]), **kw) for s in range(len(scs))]
    assert all(h.dims.threads == mixed.dims.threads for h in homo)
    for h in homo:          # the float32 raster is chosen per batch, from its widest source: the same kernel for both
        h.dims.obs_sigma_cells = mixed.dims.obs_sigma_cells
    rng = np.random.default_rng(11)
    acts = rng.uniform(0.0, 1.0, size=(steps, B, 3))
    acts[..., 2] *= 0.1
    w = (1.0, 1.0, -10.0, 1.0)
    envs = [mixed] + homo
    obs32 = [torch.zeros((e.B, 4, e.S, e.S), dtype=torch.float32, device=e.device) for e in envs]
    act = [torch.zeros((e.B, 3), dtype=torch.float64, device=e.device) for e in envs]
    for e, o in zip(envs, obs32):
        e.reset()
        if controller:
            e.get_state(out=o)
    for k in range(steps):
        for j, e in enumerate(envs):
            if controller:                                   # the RandomController law, decoded on the device
                e.linear_controller_action(obs32[j], w, out=act[j])
                e.rollout_step(act[j], obs32[j])
            else:
                a = acts[k] if j == 0 else acts[k][rows[j - 1]]
                e.rollout_step(torch.as_tensor(a, device=e.device))
        if controller:
            for s in range(len(scs)):
                assert _same(act[0][torch.as_tensor(rows[s], device=mixed.device)], act[s + 1]), (k, s, "action")
        for s in range(len(scs)):
            _compare_rows(mixed, homo[s], rows[s], (k, s), obs=(k % obs_every == 0))
    assert float(_np(mixed.hdr("ERR")).max()) == 0.0
    return mixed.counters()


@pytest.mark.parametrize("budget,rounds", [(0, 0), (60, 0), (60, 2)])
@pytest.mark.parametrize("kind,threads", [("small", 32), ("large", 64), ("golden", 64)])
def test_mixed_equals_homogeneous(dev, kind, threads, budget, rounds):
    cnt = _check_mixed_equals_homogeneous(dev, _scenarios(kind), B=10, steps=40, threads=threads, budget=budget, rounds=rounds)
    assert cnt["decisions"] > 100


@pytest.mark.gpu
@pytest.mark.parametrize("kind,threads", [("small", 32), ("large", 64)])
def test_mixed_equals_homogeneous_reordered_launch(dev, kind, threads):
    """2304 rows in one launch: k_step_order reorders the mixed batch's CTAs (longest step first), not the smaller ones'."""
    if dev == "cpu":
        pytest.skip("launch order exists on the GPU only")
    _check_mixed_equals_homogeneous(dev, _scenarios(kind), B=2304, steps=25, threads=threads, budget=60, rounds=0, obs_every=8)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,threads", [("small", 32), ("golden", 64)])
def test_mixed_equals_homogeneous_random_controller(dev, kind, threads):
    if dev == "cpu":
        pytest.skip("the emulation has no density-map decoder")
    cnt = _check_mixed_equals_homogeneous(dev, _scenarios(kind), B=64, steps=30, threads=threads, budget=0, rounds=0,
                                          controller=True)
    assert cnt["decisions"] > 500


def test_charge_rates_leave_padding_nodes_alone(dev):
    """wrsn_k_charge on a mixed batch whose smaller scenarios' padding nodes are alive, with a charger on top of them (the
    scenario record holds them at the origin): each row's rates are the reference's over its own nodes, and the padding columns
    of node_rate keep what the caller put there."""
    from oracle.wrsn_oracle import charge_rates_reference
    gs, env = _golden_batch(("ep_basic_n50", "ep_full_n100", "ep_full_n200"), dev)      # 82 / 98 / 132 nodes
    env.reset()
    E, sid, Ns = env.E, _np(env.scen_id), _np(env.num_nodes)
    assert Ns.min() < env.N
    env.view("status")[:] = 1                                      # padding columns included
    mc = env.view("mc")
    for b in range(env.B):
        nodes = env.scenarios[sid[b]].nodes
        mc[b, 0, E["WRSN_MC_X"]], mc[b, 0, E["WRSN_MC_Y"]] = 0.0, 0.0
        for a in range(1, env.M):                                  # a few metres off a node: several nodes within range
            mc[b, a, E["WRSN_MC_X"]], mc[b, a, E["WRSN_MC_Y"]] = float(nodes[7 * a][0]) + 3.0, float(nodes[7 * a][1]) - 2.0
    sentinel = -7.25
    out = (torch.full((env.B, env.N), sentinel, dtype=torch.float64, device=env.device),
           torch.zeros((env.B, env.M), dtype=torch.float64, device=env.device))
    node_rate, mc_rate = (_np(t) for t in env.charge_rates(out=out))
    status, mx, my, mcp = _np(env.view("status")), _np(env.mc("X")), _np(env.mc("Y")), env.mc_type
    for b in range(env.B):
        N = int(Ns[b])
        rr, cr = charge_rates_reference(env.scenarios[sid[b]].nodes, status[b, :N], np.stack([mx[b], my[b]], 1), np.ones(env.M),
                                        mcp["charging_range"], mcp["alpha"], mcp["beta"])
        assert (rr != 0).sum() >= 2 and (cr[1:] != 0).all(), b
        np.testing.assert_allclose(node_rate[b, :N], rr, rtol=1e-14, atol=0, err_msg=str(b))
        np.testing.assert_allclose(mc_rate[b], cr, rtol=1e-14, atol=0, err_msg=str(b))
        assert (node_rate[b, N:] == sentinel).all(), b


# ------------------------------------------------------------------ 3. against the C oracle
def test_mixed_vs_oracle(dev):
    scs = [synthetic(num_nodes=40, num_targets=120, seed=3, num_gateways=2), synthetic(num_nodes=60, num_targets=70, seed=11),
           synthetic(num_nodes=100, num_targets=50, seed=12)]
    B, steps = 6, 40
    env = BatchedWRSN(scs, num_agent=3, num_envs=B, device=dev)
    sid = _np(env.scen_id)
    Ns, Ts = _np(env.num_nodes), _np(env.num_targets)
    assert list(Ns) == [scs[s].N for s in sid] and list(Ts) == [scs[s].T for s in sid]
    rng = np.random.default_rng(5)
    acts = rng.uniform(0.0, 1.0, size=(steps, B, 3))
    acts[..., 2] *= 0.1
    oracles = [OracleWRSN(scenario_from_dict(scs[sid[b]].to_dict()), num_agent=3) for b in range(B)]
    for o in oracles:
        o.set_event_budget(3_000_000)
    req = env.reset()
    oreq = [o.reset() for o in oracles]
    live = np.ones(B, bool)
    n_dec = 0
    for k in range(steps + 1):
        aid = _np(req.agent_id)
        status, level, energy, tact = _np(env.view("status")), _np(env.view("level")), _np(env.view("energy")), _np(env.targets_active())
        for b in range(B):
            if not live[b]:
                continue
            r, o, N, tag = oreq[b], oracles[b], int(Ns[b]), (b, k)
            nd = o.nodes()
            assert int(aid[b]) == r["raw_agent_id"] and int(_np(req.terminal)[b]) == int(r["terminal"]), tag
            assert float(_np(req.now)[b]) == r["now"], tag
            assert np.array_equal(status[b, :N], nd["status"]) and not status[b, N:].any(), tag
            assert np.array_equal(level[b, :N].astype(np.int32), nd["level"]), tag
            assert np.array_equal(tact[b, :int(Ts[b])], o.targets_active()) and not tact[b, int(Ts[b]):].any(), tag
            np.testing.assert_allclose(energy[b, :N], nd["energy"], rtol=pc.E_RTOL, err_msg=str(tag))
            mcs = o.mcs()
            np.testing.assert_allclose(_np(env.mc("ENERGY"))[b], mcs["energy"], rtol=pc.E_RTOL, err_msg=str(tag))
            assert np.array_equal(_np(env.mc("STATUS"))[b].astype(np.uint8), mcs["status"]), tag
            if r["raw_agent_id"] >= 0:
                n_dec += 1
                if k > 0:
                    np.testing.assert_allclose(float(_np(req.reward)[b]), r["reward"], rtol=1e-9, atol=1e-18, err_msg=str(tag))
        if k == steps:
            break
        live &= aid >= 0
        if not live.any():
            break
        req = env.step(np.where(live, aid, -1).astype(np.int32), acts[k], mask=torch.as_tensor(live.astype(np.uint8)))
        for b in range(B):
            if live[b]:
                oreq[b] = oracles[b].step(int(aid[b]), acts[k][b])
    assert float(_np(env.hdr("ERR")).max()) == 0.0
    assert n_dec > 100


# ------------------------------------------------------------------ 4. shards of a mixed batch == the whole batch
def test_mixed_shards_equal_whole(dev):
    scs = [synthetic(num_nodes=40, num_targets=60, seed=31), synthetic(num_nodes=90, num_targets=40, seed=32),
           synthetic(num_nodes=70, num_targets=110, seed=33)]
    pc.check_sharded_equals_unsharded(scs, dev, num_envs=7, steps=30, seed=2, world=2)
    pc.check_sharded_equals_unsharded(scs, dev, num_envs=7, steps=30, seed=2, world=3, budget=20, rounds=2)


# ------------------------------------------------------------------ 5. API
def _expected_dims(N, T):
    threads, per = 32, (N + 3) // 4
    while threads < per and threads < 128:
        threads *= 2
    if N > 9 * threads:
        threads = 256
    return dict(Npad=(N + 15) // 16 * 16, W=(N + 31) // 32, Tw=max((T + 31) // 32, 1), threads=threads)


def test_dims_and_counts(dev):
    # a homogeneous batch: the dims of its one size, as before mixed sizes existed
    for n, t in ((100, 100), (60, 70), (150, 170)):
        scs = [synthetic(num_nodes=n, num_targets=t, seed=s, num_gateways=4) for s in (1, 2)]
        env = BatchedWRSN(scs, num_agent=3, num_envs=4, device=dev)
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = 4, n, t, 3, 100, env.dims.Emax, env.dims.TEmax, 2
        assert env.L.wrsn_dims_finalize(ctypes.byref(d)) == 0
        want = _expected_dims(n, t)
        got = {k: getattr(env.dims, k) for k in want}
        assert got == want and env.dims.state_bytes == d.state_bytes and env.dims.smem_bytes == d.smem_bytes, (n, t)
        assert (env.N, env.T) == (n, t) and _np(env.num_nodes).tolist() == [n] * 4 and _np(env.num_targets).tolist() == [t] * 4
    # a mixed batch: dims of the largest counts, each row's own counts, views of the largest width
    gs, env = _golden_batch(GOLDEN_MIXED, dev)
    assert _np(env.num_nodes).tolist() == [82, 82, 82, 98, 132] and _np(env.num_targets).tolist() == [50, 50, 50, 100, 200]
    assert env.num_nodes.dtype == torch.int32 and env.num_nodes.device == env.device and env.num_targets.dtype == torch.int32
    assert (env.N, env.T) == (132, 200)
    assert {k: getattr(env.dims, k) for k in ("Npad", "W", "Tw", "threads")} == _expected_dims(132, 200)
    env.reset()
    assert tuple(env.view("energy").shape) == (5, 132) and tuple(env.targets_active().shape) == (5, 200)
    assert tuple(env.get_network_fitness()[0].shape) == (5, 200) and tuple(env.charge_rates()[0].shape) == (5, 132)
    sid = np.array([4, 0, 3, 3, 1])
    env = BatchedWRSN([pc.sc_from_golden(g) for g in gs], num_agent=3, mc_type=mc_dict_of(gs[0]), scenario_index=sid, device=dev)
    assert _np(env.num_nodes).tolist() == [132, 82, 98, 98, 82]
    # the charger count is one number for the whole batch: there is no way to give scenarios different ones
    with pytest.raises(TypeError):
        BatchedWRSN([pc.sc_from_golden(g) for g in gs[:2]], num_agent=[3, 2], device=dev)


# ------------------------------------------------------------------ 6. training across sizes
@pytest.mark.gpu
def test_ippo_iteration_on_a_mixed_batch(dev, tmp_path):
    """One BatchedIPPO iteration (U-Net actors, CNN critics, density maps decoded on the device) over the five golden sizes."""
    if dev == "cpu":
        pytest.skip("the U-Net trainer runs on the GPU")
    from multi_agent_rl_wrsn_b200 import BatchedIPPO
    torch.manual_seed(0)
    args = dict(seed=0, lr=3.0e-4, gamma=0.99, clip=0.2, batch_size=64, n_updates_per_iteration=2, save_freq=1, gae=True,
                norm_adv=True, minibatch_size=32, ent_coef=0.0, vf_coef=0.5, gae_lambda=0.95, max_grad_norm=0.5, clip_vloss=True)
    gs = [golden(n) for n in GOLDEN_MIXED]
    env = BatchedWRSN([pc.sc_from_golden(g) for g in gs], num_agent=3, mc_type=mc_dict_of(gs[0]), num_envs=100, device=dev,
                      step_budget=60)
    gen = torch.Generator(device=dev).manual_seed(1)
    t = BatchedIPPO(args, env, window=4, generator=gen)
    hist = t.train(0, str(tmp_path / "save"))
    assert len(hist) == 3 and all(np.isfinite(h["loss"]) and np.isfinite(h["approx_kl"]) for h in hist)
    assert min(t.last_rollout["transitions"]) >= 64
    env.raise_on_error()
    assert float(env.hdr("ERR").max()) == 0.0
