"""Copies of running environments: BatchedWRSN.fork, snapshot / restore and EnvSnapshot files (wrsn_copy_rows).

Episodes are deterministic functions of their actions (SURVEY Q8), so a copied row is checked exactly: it must continue, byte for
byte, as a fresh batch that replays its whole action history from reset.  Each check runs on the host emulation of the kernel
source and (``-m gpu``) on the sm_100a kernels; a snapshot taken on the GPU must continue under the host build as well."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, EnvSnapshot, _lib, synthetic
from multi_agent_rl_wrsn_b200.sharding import shard_range, shard_scenario_index
from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO, golden, mc_dict_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
BACKENDS = ["cpu", pytest.param(GPU, marks=pytest.mark.gpu)]
GOLDEN3 = ("ep_basic_n50", "ep_full_n100", "ep_full_n200")      # 82 / 98 / 132 nodes
W_RANDOM = (1.0, 1.0, -10.0, 1.0)                               # the reference's RandomController as a linear map of the channels


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


_VIEWS = ("energy", "rr", "cs", "esend", "logc", "nbef", "naft", "level", "parent", "status", "logtick", "ring",
          "hdr", "mc", "proc", "tact_words", "conn_words")
_REQ = ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats", "sticky")


def _golden_scenarios(names=GOLDEN3):
    gs = [golden(n) for n in names]
    return [pc.sc_from_golden(g) for g in gs], mc_dict_of(gs[0])


def _acts(steps, B, seed):
    a = np.random.default_rng(seed).uniform(0.0, 1.0, size=(steps, B, 3))
    a[..., 2] *= 0.1
    return a


def _compare(a, ra, b, rb, tag, obs=True):
    """Rows ra of batch a against rows rb of batch b (the same scenarios, possibly at other indices): the request rows, every
    typed view of the records, the fitness and the float64 observation."""
    ra, rb = torch.as_tensor(ra, device=a.device), torch.as_tensor(rb, device=b.device)
    for f in _REQ:
        assert _same(getattr(a.req, f)[ra], getattr(b.req, f)[rb]), (tag, f)
    for f in _VIEWS:
        assert _same(a.view(f)[ra], b.view(f)[rb]), (tag, f)
    end = int(a._foff[a.E["WRSN_F_SCRATCH"]])
    assert torch.equal(a.state[ra, :end], b.state[rb, :end]), tag
    assert torch.equal(a.num_nodes[ra], b.num_nodes[rb]) and torch.equal(a.num_targets[ra], b.num_targets[rb]), tag
    fa, fb = a.get_network_fitness(), b.get_network_fitness()
    assert _same(fa[0][ra], fb[0][rb]) and _same(fa[1][ra], fb[1][rb]), tag
    if obs:
        assert _same(a.get_state(dtype=torch.float64)[ra], b.get_state(dtype=torch.float64)[rb]), tag


# ------------------------------------------------------------------ 1. fork == replay
def _fork_equals_replay(device, B, k, steps, budget, rounds, controller=False, obs_every=5):
    scs, mc = _golden_scenarios()
    sid = np.random.default_rng(3).permutation(np.arange(B) % len(scs)).astype(np.int32)
    kw = dict(num_agent=3, mc_type=mc, device=device, step_budget=budget, step_rounds=rounds)
    env = BatchedWRSN(scs, num_envs=B, scenario_index=sid, **kw)
    acts = _acts(k + steps + 40, B, seed=B + k)
    obs = torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=env.device)
    act = torch.zeros((B, 3), dtype=torch.float64, device=env.device)

    def advance(e, t, rows_of_stream):
        if controller:                                   # the RandomController law, decoded on the device
            e.linear_controller_action(obs_of[id(e)], W_RANDOM, out=act_of[id(e)])
            e.rollout_step(act_of[id(e)], obs_of[id(e)])
        else:
            e.rollout_step(torch.as_tensor(acts[t][rows_of_stream], device=e.device))

    obs_of, act_of = {id(env): obs}, {id(env): act}
    env.reset()
    if controller:
        env.get_state(out=obs)
    for t in range(k):
        advance(env, t, np.arange(B))
    while budget and not (env.req.agent_id == -4).any():          # fork with a step in flight
        advance(env, k, np.arange(B))
        k += 1
        assert k < 40
    # sources: rows in flight first, then the others; destinations: the other rows, a third of the batch
    aid = _np(env.req.agent_id)
    order = np.concatenate([np.nonzero(aid == -4)[0], np.nonzero(aid != -4)[0]])
    n = B // 3
    src, dst = order[:n], order[n:2 * n]
    if budget:
        assert (aid[src] == -4).any(), "no source row is in flight at the fork"
    assert (sid[src] != sid[dst]).any(), "every destination already had its source's scenario"
    env.fork(src, dst)
    if controller:
        env.get_state(out=obs)                           # the destinations' observations follow their new state
    origin = np.arange(B)
    origin[dst] = src
    replay = BatchedWRSN(scs, num_envs=B, scenario_index=sid[origin], **kw)
    obs_of[id(replay)] = torch.zeros_like(obs)
    act_of[id(replay)] = torch.zeros_like(act)
    replay.reset()
    if controller:
        replay.get_state(out=obs_of[id(replay)])
    for t in range(k):
        advance(replay, t, origin)
    _compare(env, np.arange(B), replay, np.arange(B), ("fork", k))
    for t in range(k, k + steps):
        advance(env, t, np.arange(B))
        advance(replay, t, np.arange(B))
        _compare(env, np.arange(B), replay, np.arange(B), t, obs=(t - k) % obs_every == 0)
    assert float(_np(env.hdr("ERR")).max()) == 0.0
    return env


@pytest.mark.parametrize("budget,rounds", [(0, 0), (60, 0), (60, 2)])
def test_fork_equals_replay(dev, budget, rounds):
    env = _fork_equals_replay(dev, B=12, k=9, steps=30, budget=budget, rounds=rounds)
    assert env.counters()["decisions"] > 100


@pytest.mark.gpu
def test_fork_equals_replay_reordered_launch(dev):
    """2304 rows: k_step_order reorders the launch of both batches (longest step first), each by its own records."""
    if dev == "cpu":
        pytest.skip("launch order exists on the GPU only")
    _fork_equals_replay(dev, B=2304, k=12, steps=20, budget=60, rounds=0, obs_every=10)


@pytest.mark.gpu
def test_fork_equals_replay_random_controller(dev):
    if dev == "cpu":
        pytest.skip("the emulation has no density-map decoder")
    env = _fork_equals_replay(dev, B=96, k=10, steps=25, budget=0, rounds=0, controller=True)
    assert env.counters()["decisions"] > 500


# ------------------------------------------------------------------ 2. across a death tick
def test_fork_across_a_death_tick(dev):
    """hanoi1000n200 loses its first node at 518.5 s.  Chargers that never charge leave that death where it is: a row forked
    between 300 s and that tick crosses it in the continuation (on a small budget: steps in flight), and must still equal the
    replay."""
    sc = pc.sc_from_golden(golden("net_hanoi1000n200"))
    B, budget = 4, 15
    kw = dict(num_agent=3, device=dev, step_budget=budget)
    acts = _acts(600, B, seed=5)
    acts[..., 2] = 0.0
    env = BatchedWRSN([sc], num_envs=B, **kw)
    env.reset()
    k = 0
    while float(env.now[0]) < 300.0:
        env.rollout_step(torch.as_tensor(acts[k], device=env.device))
        k += 1
        assert k < 300
    assert float(env.now[0]) < 518.5 and not torch.equal(env.state[0], env.state[2])
    src, dst = np.array([0]), np.array([2])
    env.fork(src, dst)
    replay = BatchedWRSN([sc], num_envs=B, **kw)
    replay.reset()
    for j in range(k):
        replay.rollout_step(torch.as_tensor(acts[j][[0, 1, 0, 3]], device=replay.device))
    E = env.E
    slow = [E["WRSN_H_NSLOW"], E["WRSN_H_NSPLIT"]]
    before = _np(env.view("hdr"))[:, slow]
    t = k
    while not (_np(env.view("hdr"))[:, slow][dst] > before[dst]).all():
        for e in (env, replay):
            e.rollout_step(torch.as_tensor(acts[t], device=e.device))
        _compare(env, np.arange(B), replay, np.arange(B), t, obs=False)
        t += 1
        assert t < len(acts)
    assert t > k + 1
    _compare(env, np.arange(B), replay, np.arange(B), "after the death tick")
    assert float(_np(env.hdr("ERR")).max()) == 0.0


# ------------------------------------------------------------------ 3. save -> load -> restore
def test_save_load_restore_continues_the_run(dev, tmp_path):
    """Restore into a fresh batch of another size, at permuted rows, with the scenario list permuted: the continuation equals the
    uninterrupted run byte for byte."""
    scs, mc = _golden_scenarios()
    B, k, steps = 9, 8, 25
    kw = dict(num_agent=3, mc_type=mc, device=dev, step_budget=60)
    run = BatchedWRSN(scs, num_envs=B, **kw)
    acts = _acts(k + steps, B, seed=17)
    run.reset()
    for t in range(k):
        run.rollout_step(torch.as_tensor(acts[t], device=run.device))
    snap = run.snapshot()
    assert len(snap) == B and _np(snap.ids).tolist() == list(range(B))
    snap.save(str(tmp_path / "rows.pt"))
    loaded = EnvSnapshot.load(str(tmp_path / "rows.pt"))
    assert loaded.device.type == "cpu" and loaded.meta == snap.meta
    perm = [2, 0, 1]
    target = BatchedWRSN([scs[p] for p in perm], num_envs=13, **kw)
    target.reset()
    rows = np.random.default_rng(1).permutation(13)[:B]
    target.restore(loaded, rows=rows)
    assert _np(target.scen_id)[rows].tolist() == [perm.index(s) for s in _np(run.scen_id)]
    _compare(run, np.arange(B), target, rows, "restored")
    for t in range(k, k + steps):
        run.rollout_step(torch.as_tensor(acts[t], device=run.device))
        a = np.zeros((13, 3))
        a[rows] = acts[t]
        target.rollout_step(torch.as_tensor(a, device=target.device))
        _compare(run, np.arange(B), target, rows, t, obs=t % 5 == 0)
    # select: rows by global id, in the order asked
    part = loaded.select([5, 1])
    assert _np(part.ids).tolist() == [5, 1] and torch.equal(part.state[0], loaded.state[5])


# ------------------------------------------------------------------ 4. resharding
def test_reshard_two_ways_into_three(dev):
    """Snapshot a job split over two shards, restore it into three shards, continue: every shard equals its block of the whole
    batch run without a stop."""
    scs = [synthetic(num_nodes=40, num_targets=60, seed=31), synthetic(num_nodes=90, num_targets=40, seed=32),
           synthetic(num_nodes=70, num_targets=110, seed=33)]
    n, k, steps = 7, 10, 25
    kw = dict(num_agent=3, device=dev, step_budget=20, step_rounds=2)
    acts = _acts(k + steps, n, seed=2)

    def shards(world):
        out = []
        for r in range(world):
            lo, hi = shard_range(n, r, world)
            out.append((lo, hi, BatchedWRSN(scs, num_envs=hi - lo, scenario_index=shard_scenario_index(n, len(scs), r, world), **kw)))
        return out

    whole = shards(1)[0][2]
    whole.reset()
    two = shards(2)
    for _, _, p in two:
        p.reset()
    for t in range(k):
        whole.rollout_step(torch.as_tensor(acts[t], device=whole.device))
        for lo, hi, p in two:
            p.rollout_step(torch.as_tensor(acts[t, lo:hi], device=p.device))
    snap = EnvSnapshot.cat([p.snapshot(base=lo) for lo, _, p in two])
    assert sorted(_np(snap.ids).tolist()) == list(range(n))
    three = shards(3)
    for lo, hi, p in three:
        p.restore(snap, base=lo)
    for t in range(k, k + steps):
        whole.rollout_step(torch.as_tensor(acts[t], device=whole.device))
        for lo, hi, p in three:
            p.rollout_step(torch.as_tensor(acts[t, lo:hi], device=p.device))
            _compare(whole, np.arange(lo, hi), p, np.arange(hi - lo), (t, lo), obs=t % 5 == 0)


# ------------------------------------------------------------------ 5. refusals
def _small(device, num_agent=3, map_size=100, scs=None, B=4):
    scs = scs or [synthetic(num_nodes=100, num_targets=100, seed=1), synthetic(num_nodes=40, num_targets=40, seed=2),
                  synthetic(num_nodes=40, num_targets=40, seed=3)]
    env = BatchedWRSN(scs, num_agent=num_agent, map_size=map_size, num_envs=B, device=device)
    env.reset()
    return env


def test_restore_refuses_what_it_cannot_continue(dev, tmp_path):
    env = _small(dev)
    snap = env.snapshot()
    with pytest.raises(ValueError, match="dims.M"):
        _small(dev, num_agent=2).restore(snap)
    with pytest.raises(ValueError, match="dims.S"):
        _small(dev, map_size=50).restore(snap)
    # the same layout (the 100-node scenario sets every maximum), but the third scenario replaced by another
    other = _small(dev, scs=[synthetic(num_nodes=100, num_targets=100, seed=1), synthetic(num_nodes=40, num_targets=40, seed=2),
                             synthetic(num_nodes=40, num_targets=40, seed=4)])
    assert [getattr(other.dims, f) for f in ("N", "T", "Emax", "TEmax")] == [getattr(env.dims, f) for f in ("N", "T", "Emax", "TEmax")]
    with pytest.raises(ValueError, match="fingerprints"):
        other.restore(snap)
    other.restore(snap.select([0, 1]), rows=[3, 2])      # rows of the scenarios both batches have are fine
    # a file whose ABI version was edited
    path = str(tmp_path / "s.pt")
    snap.save(path)
    d = torch.load(path, weights_only=True)
    d["meta"]["abi"] = d["meta"]["abi"] - 1
    torch.save(d, path)
    with pytest.raises(ValueError, match="abi"):
        env.restore(EnvSnapshot.load(path))
    # lengths and indices
    with pytest.raises(ValueError, match="rows"):
        env.restore(snap, rows=[0, 1])
    with pytest.raises(ValueError, match="rows"):
        env.restore(snap, rows=[0, 1, 2, 4])
    with pytest.raises(ValueError, match="rows"):
        env.restore(snap, rows=[0, 1, 1, 2])
    with pytest.raises(ValueError, match="rows"):
        env.restore(EnvSnapshot.cat([snap, snap]))        # every global id twice


def test_fork_refuses_bad_rows(dev):
    env = _small(dev)
    before = env.state.clone()
    for src, dst, what in (([0, 1], [2, 2], "distinct"), ([0, 1], [1, 2], "also in src"), ([0], [4], r"\[0, 4\)"),
                           ([-1], [2], r"\[0, 4\)"), ([0, 1], [2], "same length")):
        with pytest.raises(ValueError, match=what):
            env.fork(src, dst)
    assert torch.equal(env.state, before)


def test_raw_copy_skips_out_of_range_pairs(dev):
    """wrsn_copy_rows itself: a pair with an index outside [0, src_B) / [0, dst_B) is skipped, leaving both buffers as they were."""
    env = _small(dev)
    snap = env.snapshot()
    snap.state.fill_(7)
    keep = (env.state.clone(), env.req.now.clone(), env.scen_id.clone(), snap.state.clone(), snap.req["now"].clone(), snap.scen.clone())
    from multi_agent_rl_wrsn_b200.snapshot import c_request
    src = torch.tensor([env.B, -1, 0, 1], dtype=torch.int32, device=env.device)
    dst = torch.tensor([0, 1, env.B, -2], dtype=torch.int32, device=env.device)
    sq = c_request(snap.req)
    rc = env.L.wrsn_copy_rows(ctypes.byref(env.dims), 4, snap.state.data_ptr(), ctypes.byref(sq), snap.scen.data_ptr(), src.data_ptr(),
                              len(snap), env.state.data_ptr(), ctypes.byref(env.req.c), env.scen_id.data_ptr(), dst.data_ptr(), env.B, None)
    if dev != "cpu":
        torch.cuda.synchronize()
    assert rc == 0
    after = (env.state, env.req.now, env.scen_id, snap.state, snap.req["now"], snap.scen)
    assert all(torch.equal(a, b) for a, b in zip(keep, after))


def test_copy_rows_checks_equal_in_both_libraries(emu_built):
    """The argument checks live in the shared host side of the ABI: both libraries refuse the same inputs with the same message
    (nothing passes the checks here, so nothing is launched)."""
    import __graft_entry__ as g
    g.build()
    libs = [_lib._bind(ctypes.CDLL(_lib.LIB_PATH)), _lib._bind(ctypes.CDLL(os.path.join(EMU_DIR, "libwrsn_emu.so")))]
    B = 2

    def call(L, finalize=True, n=1, src_B=B, dst_B=B, null=None, null_req=None):
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = B, 50, 50, 3, 100, 300, 100, 1
        if finalize:
            assert L.wrsn_dims_finalize(ctypes.byref(d)) == 0
        bufs = dict(state=np.zeros(max(d.state_bytes, 16) * B, np.uint8), scen_id=np.zeros(B, np.int32), rows=np.zeros(B, np.int32))
        req = {f: np.zeros(B * 3, np.float64) for f in ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats", "sticky")}
        p = {k: (None if k == null else a.ctypes.data) for k, a in bufs.items()}
        q = _lib.Request(*[(None if f == null_req else req[f].ctypes.data) if f in req else None for f, _ in _lib.Request._fields_])
        rc = L.wrsn_copy_rows(ctypes.byref(d), n, p["state"], ctypes.byref(q), p["scen_id"], p["rows"], src_B,
                              p["state"], ctypes.byref(q), p["scen_id"], p["rows"], dst_B, None)
        return rc, L.wrsn_last_error()

    cases = [(dict(finalize=False), b"dims not finalized"), (dict(n=-1), b"must not be negative"), (dict(src_B=0), b"both must be positive"),
             (dict(dst_B=-3), b"both must be positive"), (dict(null="state"), b"is NULL"), (dict(null="rows"), b"is NULL"),
             (dict(null="scen_id"), b"is NULL"), (dict(null_req="flags"), b"must not be NULL"),
             (dict(null_req="agent_id"), b"must not be NULL")]
    for kw, msg in cases:
        got = [call(L, **kw) for L in libs]
        assert got[0] == got[1], (kw, got)
        assert got[0][0] == -1 and msg in got[0][1], (kw, got)
    assert [call(L, n=0)[0] for L in libs] == [0, 0]                        # n == 0: nothing to do


# ------------------------------------------------------------------ 6. GPU -> host build
@pytest.mark.gpu
def test_gpu_snapshot_continues_under_the_host_build(emu_built, tmp_path):
    """A mid-episode snapshot of a RandomController rollout on the device, saved, loaded and restored under the host build: both
    continue with the same uniform actions.  Every field outside update_reward's outputs is equal byte for byte; reward, detail
    and the chargers' exclusive reward agree to 1e-9 (the host build computes 1/x exactly where the device uses rcp.approx +
    Newton, DESIGN §4.1)."""
    helpers.use_cuda_build()
    scs, mc = _golden_scenarios()
    B, k, steps = 256, 12, 30
    kw = dict(num_agent=3, mc_type=mc, step_budget=60)
    env = BatchedWRSN(scs, num_envs=B, device=GPU, **kw)
    obs = torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=env.device)
    act = torch.zeros((B, 3), dtype=torch.float64, device=env.device)
    env.reset()
    env.get_state(out=obs)
    for _ in range(k):
        env.linear_controller_action(obs, W_RANDOM, out=act)
        env.rollout_step(act, obs)
    assert (_np(env.req.stats)[:, 2] >= 1).all()
    path = str(tmp_path / "gpu_rows.pt")
    env.snapshot().save(path)
    acts = _acts(steps, B, seed=23)
    E = env.E
    excl = E["WRSN_MC_EXCL"]

    def record(e):
        mcv = _np(e.view("mc"))
        out = dict(req={f: _np(getattr(e.req, f)) for f in _REQ}, excl=mcv[:, :, excl].copy())
        mcv[:, :, excl] = 0.0
        mc_bytes = mcv.view(np.uint8)
        st = _np(e.state)
        lo, hi = int(e._foff[E["WRSN_F_MC"]]), int(e._foff[E["WRSN_F_MC"]]) + mc_bytes.shape[1] * mc_bytes.shape[2]
        st[:, lo:hi] = mc_bytes.reshape(B, -1)
        out["state"] = st[:, :int(e._foff[E["WRSN_F_SCRATCH"]])]
        return out

    dev_run = []
    for t in range(steps):
        env.rollout_step(torch.as_tensor(acts[t], device=env.device))
        dev_run.append(record(env))
    env.raise_on_error()
    try:
        helpers.use_host_build()
        host = BatchedWRSN(scs, num_envs=B, device="cpu", **kw)
        host.restore(EnvSnapshot.load(path))
        for t in range(steps):
            host.rollout_step(torch.as_tensor(acts[t]))
            got, want = record(host), dev_run[t]
            assert np.array_equal(got["state"], want["state"]), t
            for f in _REQ:
                g, w = got["req"][f], want["req"][f]
                if f in ("reward", "detail"):
                    assert np.array_equal(np.isnan(g), np.isnan(w)), (t, f)
                    np.testing.assert_allclose(g, w, rtol=1e-9, atol=0, equal_nan=True, err_msg=str((t, f)))
                else:
                    assert np.array_equal(g, w, equal_nan=g.dtype.kind == "f"), (t, f)
            np.testing.assert_allclose(got["excl"], want["excl"], rtol=1e-9, atol=1e-300, err_msg=str(t))
    finally:
        helpers.use_cuda_build_lazy()
