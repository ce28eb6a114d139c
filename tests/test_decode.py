"""Density-map action decode (SURVEY 8f-1): ``wrsn_decode_density_map`` (CUDA) against the CPU restatement of
``WRSN.density_map_to_action`` (oracle/decode_oracle.py), and that restatement against the reference's golden actions."""
import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, Scenario, _lib, synthetic
from oracle import decode_oracle as do
from oracle.wrsn_oracle import OracleWRSN, scenario_from_dict
from tests import helpers, parity_cases as pc
from tests.helpers import golden, mc_dict_of

DEV = "cuda:0"


def _mc_default():
    from multi_agent_rl_wrsn_b200.scenario import load_mc_type
    return load_mc_type(None)


def test_decode_oracle_matches_reference_golden():
    """The decode restatement, fed with the C oracle's observations (RandomController rule s0 + s1 - 10 s2 + s3,
    runner/checkRL.py), reproduces the actions the unmodified reference decoded (dmap_random_n50.npz)."""
    g = golden("dmap_random_n50")
    sc = pc.sc_from_golden(g)
    mc = _mc_default()
    o = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=int(g["num_agent"]))
    r = o.reset()
    frame = o.consts()["frame"]
    xy = np.asarray(sc.nodes, np.float64).reshape(-1, 2)
    thr = float(g["sc_par"][1])
    for i in range(int(g["n"])):
        assert r["raw_agent_id"] == int(g["fed_agent"][i])
        st = r["state"]
        dm = do.normalise_map(np.copy(st[0] + st[1] - 10 * st[2] + st[3]))
        nd = o.nodes()
        act = do.density_map_to_action(dm, frame, xy, nd["status"], nd["energy"], nd["cs"], thr, mc["charging_range"],
                                       mc["alpha"], mc["beta"], 100)
        np.testing.assert_allclose(act, g["action"][i], rtol=1e-6, atol=1e-9)
        r = o.step(r["raw_agent_id"], np.clip(act, 0.0, 1.0))
        assert r["raw_agent_id"] == int(g["agent_id"][i])
        np.testing.assert_allclose(r["now"], float(g["now"][i]), rtol=1e-7)


def test_percentile_and_argmax_conventions():
    """Corner cases of the restated conventions the kernel mirrors: first maximum wins, ties at the percentile keep
    both values, a uniform map keeps everything."""
    S = 100
    dm = np.zeros((S, S)); dm[3, 7] = 0.5; dm[60, 2] = 0.5
    frame = np.array([0.0, 1000.0, 0.0, 1000.0])
    xy = np.zeros((1, 2)); st = np.zeros(1, np.uint8)
    a = do.density_map_to_action(dm, frame, xy, st, np.ones(1), np.ones(1), 0.0, 27.0, 4500.0, 30.0, S)
    np.testing.assert_allclose(a, [(3 + 0.5) / S, (7 + 0.5) / S, 0.5])
    u = np.full((S, S), 1.0 / (S * S))
    a = do.density_map_to_action(u, frame, xy, st, np.ones(1), np.ones(1), 0.0, 27.0, 4500.0, 30.0, S)
    np.testing.assert_allclose(a, [0.5 / S, 0.5 / S, 1.0 / (S * S)], rtol=1e-12)


@pytest.fixture()
def cuda_library():
    L = helpers.use_cuda_build()
    assert not helpers.is_host_build(L) and torch.cuda.is_available()
    yield


def _rolled_env(B, steps, seed, scale2=0.05):
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + k) for k in range(4)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=B, device=DEV)
    env.reset()
    g = torch.Generator(device=DEV); g.manual_seed(seed)
    for _ in range(steps):
        a = torch.rand((B, 3), dtype=torch.float64, device=DEV, generator=g); a[:, 2] *= scale2
        env.rollout_step(a)
    return env, scs


def _oracle_decode(env, scs, b, dm):
    st = env.statics[int(env.scen_id[b])]
    par = st["par"]
    xy = np.stack([np.asarray(st["x"]), np.asarray(st["y"])], 1)[:env.N]
    frame = np.array([par["F0"], par["F1"], par["F2"], par["F3"]])
    return do.density_map_to_action(do.normalise_map(dm), frame, xy, env.view("status")[b].cpu().numpy(),
                                    env.view("energy")[b].cpu().numpy(), env.view("cs")[b].cpu().numpy(), par["THR"],
                                    par["MC_R"], par["MC_ALPHA"], par["MC_BETA"], env.S, return_result=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_decode_matches_oracle(cuda_library, dtype):
    """Maps of three kinds (a policy-like bump near a node, the RandomController combination of the observation
    channels, raw logits that need the exp-normalisation) on rolled-out environments.
    Third component: 1e-12 (float64 maps) — it is exact arithmetic on order statistics.
    Location: identical to scipy's whenever L-BFGS-B stops at the box centre (the common case), within 1e-3 m in at
    least 90 % of the others (discontinuous objective, optimiser- and version-dependent: SURVEY 8f-1), with an objective
    value within 1e-4 relative of scipy's."""
    B = 48
    env, scs = _rolled_env(B, 60, seed=3)
    rng = np.random.default_rng(1)
    obs = env.get_state(dtype=torch.float64).cpu().numpy()
    S = env.S
    maps = np.zeros((B, S, S))
    ii = (np.arange(S) + 0.5) / S
    for b in range(B):
        kind = b % 3
        if kind == 0:
            st = env.statics[int(env.scen_id[b])]; par = st["par"]
            n = rng.integers(0, env.N)
            cx = (st["x"][n] - par["F0"]) / (par["F1"] - par["F0"]) + rng.normal(0, 0.02)
            cy = (st["y"][n] - par["F2"]) / (par["F3"] - par["F2"]) + rng.normal(0, 0.02)
            m = np.exp(-((ii[:, None] - cx) ** 2 + (ii[None, :] - cy) ** 2) / (2 * 0.03 ** 2))
            maps[b] = m / m.sum()
        elif kind == 1:
            maps[b] = obs[b][0] + obs[b][1] - 10 * obs[b][2] + obs[b][3]
        else:
            maps[b] = rng.normal(0, 2.0, (S, S))
    dm = torch.as_tensor(maps, device=DEV).to(dtype).contiguous()
    aid = env.req.agent_id.clone()
    aid[5] = -1                                       # a row without a deciding charger stays untouched
    out = torch.full((B, 3), -7.0, dtype=torch.float64, device=DEV)
    env.density_map_to_action(dm, agent_id=aid, out=out)
    got = out.cpu().numpy()
    assert np.all(got[5] == -7.0)
    host_maps = dm.cpu().numpy().astype(np.float64)
    exact, close, moved, worse = 0, 0, 0, 0
    for b in range(B):
        if int(aid[b]) < 0:
            continue
        ref, res, x0, objective = _oracle_decode(env, scs, b, host_maps[b])
        np.testing.assert_allclose(got[b, 2], ref[2], rtol=1e-12 if dtype == torch.float64 else 1e-6)
        st = env.statics[int(env.scen_id[b])]; par = st["par"]
        loc = np.array([got[b, 0] * (par["F1"] - par["F0"]) + par["F0"], got[b, 1] * (par["F3"] - par["F2"]) + par["F2"]])
        if np.array_equal(res.x, x0):                 # scipy stopped at the centre: pgtol
            np.testing.assert_allclose(got[b, :2], ref[:2], rtol=1e-14, atol=1e-15)
            exact += 1
        else:
            moved += 1
            close += int(np.hypot(*(loc - res.x)) <= 1e-3)
            worse += int(-objective(loc) < -res.fun * (1.0 - 1e-4))
    assert exact >= 10
    assert moved == 0 or (close >= 0.9 * moved and worse <= 0.1 * moved), (exact, moved, close, worse)


@pytest.mark.gpu
def test_decode_heavy_weights_track_scipy(cuda_library):
    """Nodes close to their threshold make the objective (and its gradient) large: L-BFGS-B really iterates.  The
    kernel's climb must end where scipy's does (the same cusp) in the large majority of cases."""
    B = 64
    env, scs = _rolled_env(B, 30, seed=5)
    en = env.view("energy"); thr = 540.0
    rng = np.random.default_rng(2)
    S = env.S
    ii = (np.arange(S) + 0.5) / S
    maps = np.zeros((B, S, S))
    for b in range(B):
        st = env.statics[int(env.scen_id[b])]; par = st["par"]
        n = int(rng.integers(0, env.N))
        en[b, n] = thr + 15.0                         # a node about to die: weight energyCS / (E - thr) ~ 50 x larger
        cx = (st["x"][n] - par["F0"]) / (par["F1"] - par["F0"]) + rng.normal(0, 0.015)
        cy = (st["y"][n] - par["F2"]) / (par["F3"] - par["F2"]) + rng.normal(0, 0.015)
        m = np.exp(-((ii[:, None] - cx) ** 2 + (ii[None, :] - cy) ** 2) / (2 * 0.03 ** 2))
        maps[b] = m / m.sum()
    dm = torch.as_tensor(maps, device=DEV)
    aid = torch.zeros(B, dtype=torch.int32, device=DEV)
    got = env.density_map_to_action(dm, agent_id=aid).cpu().numpy()
    moved, close = 0, 0
    for b in range(B):
        ref, res, x0, objective = _oracle_decode(env, scs, b, maps[b])
        st = env.statics[int(env.scen_id[b])]; par = st["par"]
        loc = np.array([got[b, 0] * (par["F1"] - par["F0"]) + par["F0"], got[b, 1] * (par["F3"] - par["F2"]) + par["F2"]])
        if not np.array_equal(res.x, x0):
            moved += 1
            close += int(np.hypot(*(loc - res.x)) <= 1e-3)
    assert moved >= 20 and close >= 0.85 * moved, (moved, close)


@pytest.mark.gpu
def test_decode_full_size_properties(cuda_library):
    """BASELINE config 2 size (4096 environments): one-hot maps decode to their cell centre with charge fraction 1,
    uniform maps to cell (0, 0) with 1 / S^2, and decoding is deterministic."""
    sc = synthetic(num_nodes=100, num_targets=100, seed=1)
    B = 4096
    env = BatchedWRSN(sc, num_agent=3, num_envs=B, device=DEV)
    env.reset()
    S = env.S
    g = torch.Generator(device=DEV); g.manual_seed(0)
    cell = torch.randint(0, S * S, (B,), device=DEV, generator=g)
    dm = torch.zeros((B, S * S), dtype=torch.float32, device=DEV)
    dm[torch.arange(B, device=DEV), cell] = 1.0
    env.view("status")[:] = 0                         # no alive node: the objective is flat, the centre is the answer
    a = env.density_map_to_action(dm.view(B, S, S))
    np.testing.assert_allclose(a[:, 0].cpu().numpy(), ((cell // S).double().cpu().numpy() + 0.5) / S, rtol=1e-12)
    np.testing.assert_allclose(a[:, 1].cpu().numpy(), ((cell % S).double().cpu().numpy() + 0.5) / S, rtol=1e-12)
    assert bool((a[:, 2] == 1.0).all())
    u = torch.full((B, S, S), 1.0 / (S * S), dtype=torch.float64, device=DEV)
    a = env.density_map_to_action(u)
    np.testing.assert_allclose(a[0].cpu().numpy(), [0.5 / S, 0.5 / S, 1.0 / (S * S)], rtol=1e-12)
    r = torch.rand((B, S, S), dtype=torch.float32, device=DEV, generator=g)
    assert torch.equal(env.density_map_to_action(r), env.density_map_to_action(r))


@pytest.mark.gpu
def test_linear_controller_decode_equals_materialised_map(cuda_library):
    """wrsn_decode_linear_controller (the RandomController map formed inside the decoder, channel by channel) == the decoder
    on the map torch materialises for the same expression, bit for bit, on 512 rolled-out environments."""
    B = 512
    env, scs = _rolled_env(B, 80, seed=7, scale2=0.1)
    obs = env.get_state(dtype=torch.float32)
    agents = torch.zeros(B, dtype=torch.int32, device=DEV)
    dm = obs[:, 0] + obs[:, 1] - 10.0 * obs[:, 2] + obs[:, 3]
    want = env.density_map_to_action(dm.contiguous(), agent_id=agents)
    got = env.linear_controller_action(obs, (1.0, 1.0, -10.0, 1.0), agent_id=agents)
    same = lambda x, y: bool(((x == y) | (torch.isnan(x) & torch.isnan(y))).all())   # (a map that overflows exp() decodes to a NaN
    assert same(want, got)                                                            #  charge fraction on both paths alike)
    w = (0.5, -2.0, 3.0, 0.25)                           # any weights: torch multiplies, then adds, left to right
    dm = w[0] * obs[:, 0] + w[1] * obs[:, 1] + w[2] * obs[:, 2] + w[3] * obs[:, 3]
    assert same(env.density_map_to_action(dm.contiguous(), agent_id=agents), env.linear_controller_action(obs, w, agent_id=agents))


@pytest.mark.gpu
def test_random_controller_rollout_stays_on_the_host_decode_trajectory(cuda_library):
    """How often does a RandomController rollout whose maps are decoded ON THE DEVICE leave the trajectory the reference's own
    decode (numpy + scipy's L-BFGS-B, oracle/decode_oracle.py) would have driven?  48 environments x 25 rollout steps on the
    bench's scenarios; at every decision the device's action is compared with the host decode of the same map on the same state.
    Charge fraction: 1e-6 (float32 maps).  Location: the same point within 1e-3 m in at least 90 % of the decisions (where scipy
    stops at the box centre — the common case — the device is at that centre exactly); the rest are cusps of a discontinuous
    objective where the two optimisers stop at different kinks (SURVEY 8f-1).  The counts are printed."""
    B, steps = 48, 25
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + k) for k in range(4)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=B, device=DEV)
    env.reset()
    obs = env.get_state(dtype=torch.float32)
    n_dec = n_centre = n_close = n_far = n_nan = 0
    far = []
    for k in range(steps):
        dm = (obs[:, 0] + obs[:, 1] - 10.0 * obs[:, 2] + obs[:, 3]).contiguous()
        aid = env.req.agent_id.clone()
        act = env.density_map_to_action(dm, agent_id=aid)
        got = act.cpu().numpy()
        maps = dm.cpu().numpy().astype(np.float64)
        for b in range(B):
            if int(aid[b]) < 0:
                continue
            with np.errstate(all="ignore"):
                ref, res, x0, objective = _oracle_decode(env, scs, b, maps[b])
            n_dec += 1
            if not np.isfinite(ref[2]):               # a map that overflows exp(): NaN charge fraction on both paths
                assert not np.isfinite(got[b, 2])
                n_nan += 1
                continue
            np.testing.assert_allclose(got[b, 2], ref[2], rtol=1e-6)
            par = env.statics[int(env.scen_id[b])]["par"]
            loc = np.array([got[b, 0] * (par["F1"] - par["F0"]) + par["F0"], got[b, 1] * (par["F3"] - par["F2"]) + par["F2"]])
            d = float(np.hypot(*(loc - res.x)))
            if np.array_equal(res.x, x0) and d <= 1e-9:
                n_centre += 1
            elif d <= 1e-3:
                n_close += 1
            else:
                n_far += 1
                far.append(d)
        env.rollout_step(torch.nan_to_num(act), obs)
    print("RandomController rollout, device decode against the host decode: %d decisions, %d at scipy's box centre exactly, %d within "
          "1e-3 m, %d elsewhere (median distance %.2f m), %d overflowing maps"
          % (n_dec, n_centre, n_close, n_far, float(np.median(far)) if far else 0.0, n_nan))
    assert n_dec >= B * steps // 3
    assert n_centre + n_close >= 0.9 * (n_dec - n_nan), (n_dec, n_centre, n_close, n_far, n_nan)


# ------------------------------------------------------------------ map sizes, map kinds and the decoder's edge paths
DEC_SIZES = [1, 2, 4, 7, 17, 32, 64, 100, 128, 175, 176]
DEC_MAX_S = 176                                       # the largest map whose percentile rank the decoder holds


def _rank(S):
    """R of np.percentile(., 99.9) over S * S cells (the R-th largest value is the lower interpolation point), with the
    kernel's own expression."""
    n = S * S
    return n - int(np.floor(n * 0.999 + (1.0 + 0.999 * (1.0 - 1.0 - 1.0)) - 1.0))


def _fraction_at_rank(dm, r):
    """The charge fraction of density_map_to_action with the percentile taken between the r-th and (r-1)-th largest
    values instead of the R-th and (R-1)-th."""
    flat = np.sort(dm.ravel())
    n = flat.size
    vidx = n * 0.999 + (1.0 + 0.999 * (1.0 - 1.0 - 1.0)) - 1.0
    tq = vidx - np.floor(vidx)
    lo = n - r
    a, b = flat[lo], flat[min(lo + 1, n - 1)]
    thr = a + (b - a) * tq if tq < 0.5 else b - (b - a) * (1.0 - tq)
    return dm.max() / dm.ravel()[dm.ravel() >= thr].sum()


def test_decoder_rank_limit():
    assert _rank(100) == 11 and _rank(DEC_MAX_S) == 32 and _rank(DEC_MAX_S + 1) == 33 and _rank(200) == 41


@pytest.fixture()
def host_library():
    import os
    import subprocess
    subprocess.check_call(["make", "-C", os.path.join(helpers.REPO, "tests", "emu"), "libwrsn_emu.so"], stdout=subprocess.DEVNULL)
    helpers.use_host_build()
    yield
    helpers.use_cuda_build_lazy()


def _refuses_large_maps(dev):
    for S in (DEC_MAX_S + 1, 200):
        env = BatchedWRSN(synthetic(num_nodes=40, num_targets=40, seed=2), num_agent=3, num_envs=2, map_size=S, device=dev)
        env.reset()
        aid = torch.zeros(2, dtype=torch.int32, device=env.state.device)
        with pytest.raises(RuntimeError, match=r"map_size = %d: .* up to %d" % (S, DEC_MAX_S)):
            env.density_map_to_action(torch.zeros((2, S, S), dtype=torch.float32, device=env.state.device), agent_id=aid)
        with pytest.raises(RuntimeError, match=r"map_size = %d: .* up to %d" % (S, DEC_MAX_S)):
            env.linear_controller_action(torch.zeros((2, 4, S, S), dtype=torch.float32, device=env.state.device), (1, 1, -10, 1), agent_id=aid)


def test_decoder_refuses_large_maps_host_build(host_library):
    """Both libraries share the check (wrsn_abi_host.h); the host build's decode entry points run it before they report that
    the decoder is not emulated."""
    _refuses_large_maps("cpu")
    env = BatchedWRSN(synthetic(num_nodes=40, num_targets=40, seed=2), num_agent=3, num_envs=2, map_size=DEC_MAX_S, device="cpu")
    with pytest.raises(RuntimeError, match="not available in the host emulation"):
        env.density_map_to_action(torch.zeros((2, DEC_MAX_S, DEC_MAX_S)), agent_id=torch.zeros(2, dtype=torch.int32))


@pytest.mark.gpu
def test_decoder_refuses_large_maps(cuda_library):
    _refuses_large_maps(DEV)


MAP_KINDS = ("bump", "logits", "masked", "masked_few", "ties", "onehot", "uniform")


def _make_map(kind, S, rng, cx, cy):
    ii = (np.arange(S) + 0.5) / S
    n = S * S
    if kind == "bump":                                # a distribution, at least two cells wide: on a small map a narrower
        w = max(0.03, 2.0 / S)                        # bump is one-hot in all but name, and no rank near the top shows
        m = np.exp(-((ii[:, None] - cx) ** 2 + (ii[None, :] - cy) ** 2) / (2 * w ** 2))
        return m / m.sum()
    if kind == "logits":
        return rng.normal(0, 2.0, (S, S))
    if kind in ("masked", "masked_few"):              # -inf in most cells; "few": fewer finite cells than R + 1
        m = np.full(n, -np.inf)
        k = max(1, n // 20) if kind == "masked" else max(1, min(n, _rank(S)) // 2)
        m[rng.choice(n, k, replace=False)] = rng.normal(0, 2.0, k)
        return m.reshape(S, S)
    if kind == "ties":                                # quantised: values tie at the percentile (second pass)
        return np.round(rng.uniform(0, 3, (S, S))) / 2
    if kind == "onehot":
        m = np.zeros(n); m[rng.integers(0, n)] = 1.0
        return m.reshape(S, S)
    return np.full((S, S), 1.0 / n)                   # uniform


def _locate_counts(env, got, ref, b, res, x0, counts):
    par = env.statics[int(env.scen_id[b])]["par"]
    loc = np.array([got[0] * (par["F1"] - par["F0"]) + par["F0"], got[1] * (par["F3"] - par["F2"]) + par["F2"]])
    if np.array_equal(res.x, x0):                     # scipy stopped at the centre: pgtol
        np.testing.assert_allclose(got[:2], ref[:2], rtol=1e-14, atol=1e-15)
        counts["exact"] += 1
    else:
        counts["moved"] += 1
        counts["close"] += int(np.hypot(*(loc - res.x)) <= 1e-3)
    return loc


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_decode_map_sizes_and_kinds(cuda_library, dtype):
    """Maps of seven kinds at every size from 1 x 1 to 176 x 176 against the restatement: charge fraction 1e-12 (float64 maps) /
    1e-6 (float32); location identical where scipy stops at the box centre, otherwise within 1e-3 m in at least 90 % of the
    decodes.  For every map without ties, the restatement's fraction at rank R - 1 and R + 1 differs from the one at R by more
    than the tolerance: a rank slip cannot pass."""
    rng = np.random.default_rng(17)
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    counts = dict(exact=0, moved=0, close=0)
    rank_checked = 0
    for S in DEC_SIZES:
        B = 2 * len(MAP_KINDS)
        env = BatchedWRSN(synthetic(num_nodes=100, num_targets=100, seed=1000 + S), num_agent=3, num_envs=B, map_size=S, device=DEV)
        env.reset()
        maps = []
        for b in range(B):
            st = env.statics[0]; par = st["par"]
            n = rng.integers(0, env.N)
            cx = (st["x"][n] - par["F0"]) / (par["F1"] - par["F0"]); cy = (st["y"][n] - par["F2"]) / (par["F3"] - par["F2"])
            maps.append(_make_map(MAP_KINDS[b % len(MAP_KINDS)], S, rng, cx, cy))
        dm = torch.as_tensor(np.stack(maps), device=DEV).to(dtype).contiguous()
        aid = torch.zeros(B, dtype=torch.int32, device=DEV)
        got = env.density_map_to_action(dm, agent_id=aid).cpu().numpy()
        host = dm.cpu().numpy().astype(np.float64)
        for b in range(B):
            kind = MAP_KINDS[b % len(MAP_KINDS)]
            with np.errstate(all="ignore"):
                ref, res, x0, objective = _oracle_decode(env, None, b, host[b])
            np.testing.assert_allclose(got[b, 2], ref[2], rtol=tol, err_msg=str((S, kind)))
            _locate_counts(env, got[b], ref, b, res, x0, counts)
            norm = do.normalise_map(host[b])
            R = _rank(S)
            top = np.sort(norm.ravel())[::-1][:R + 2]
            if kind in ("bump", "logits") and 2 <= R < S * S and np.unique(top).size == top.size:   # no ties near the percentile
                np.testing.assert_allclose(_fraction_at_rank(norm, R), ref[2], rtol=1e-12)
                for r in (R - 1, R + 1):          # (ranks 1 and 2 keep the same single value: below 1000 cells the
                    if 2 <= r <= S * S:           #  interpolation weight puts the percentile above the second largest)
                        assert abs(_fraction_at_rank(norm, r) - ref[2]) > tol * abs(ref[2]), (S, kind, r)
                        rank_checked += 1
    print("map sizes 1..176 (%s): %d decodes at scipy's box centre exactly, %d of %d others within 1e-3 m; %d rank slips detectable"
          % (dtype, counts["exact"], counts["close"], counts["moved"], rank_checked))
    assert counts["exact"] >= 20 and rank_checked >= 30
    assert counts["close"] >= 0.9 * counts["moved"], counts


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_decode_all_minus_inf_map(cuda_library, dtype):
    """A map that is -inf everywhere (a fully masked log-density): numpy's argmax gives cell 0, so the box is cell 0's; the
    charge fraction is NaN (0 / 0 after the normalisation) on both paths."""
    for S in (7, 100):
        B = 4
        env = BatchedWRSN(synthetic(num_nodes=100, num_targets=100, seed=1100 + S), num_agent=3, num_envs=B, map_size=S, device=DEV)
        env.reset()
        dm = torch.full((B, S, S), -float("inf"), dtype=dtype, device=DEV)
        got = env.density_map_to_action(dm, agent_id=torch.zeros(B, dtype=torch.int32, device=DEV)).cpu().numpy()
        counts = dict(exact=0, moved=0, close=0)
        for b in range(B):
            with np.errstate(all="ignore"):
                ref, res, x0, objective = _oracle_decode(env, None, b, dm[b].cpu().numpy().astype(np.float64))
            assert np.isnan(ref[2]) and np.isnan(got[b, 2])
            assert abs(got[b, 0]) <= 1.0 and abs(got[b, 1]) <= 1.0, (S, got[b])       # near cell 0, not far off the field
            _locate_counts(env, got[b], ref, b, res, x0, counts)
        assert counts["close"] == counts["moved"], counts


@pytest.mark.gpu
def test_linear_controller_rolled_path(cuda_library):
    """wrsn_decode_linear_controller with 1, 2, 3, 5 and 8 channels (the rolled path) and 4 (unrolled) == the decoder on the map
    torch forms left to right, bit for bit."""
    B, S = 64, 100
    env, scs = _rolled_env(B, 20, seed=9)
    g = torch.Generator(device=DEV); g.manual_seed(4)
    agents = torch.zeros(B, dtype=torch.int32, device=DEV)
    weights = (0.5, -2.0, 3.0, 0.25, 1.5, -0.75, 2.0, -1.25)
    same = lambda x, y: bool(((x == y) | (torch.isnan(x) & torch.isnan(y))).all())
    for C in (1, 2, 3, 4, 5, 8):
        obs = torch.randn((B, C, S, S), dtype=torch.float32, device=DEV, generator=g).contiguous()
        w = weights[:C]
        dm = w[0] * obs[:, 0]
        for c in range(1, C):
            dm = dm + w[c] * obs[:, c]
        want = env.density_map_to_action(dm.contiguous(), agent_id=agents)
        got = env.linear_controller_action(obs, w, agent_id=agents)
        assert same(want, got), C


@pytest.mark.gpu
def test_decode_locate_dense_field(cuda_library):
    """200 nodes in a 150 m square: about 120 alive nodes within reach of the box, more than the 64 the locate kernel lists in
    shared memory, so it reads the nodes from HBM.  Against scipy with the criteria above; every returned point lies in the
    box, with an objective at least the centre's."""
    rng = np.random.default_rng(3)
    nodes = rng.uniform(0, 150, (200, 2))
    sc = Scenario(nodes=nodes, targets=rng.uniform(0, 150, (50, 2)), base_station=np.array([75.0, 75.0]))
    B = 32
    env = BatchedWRSN(sc, num_agent=3, num_envs=B, device=DEV)
    env.reset()
    S = env.S
    st = env.statics[0]; par = st["par"]
    R = par["MC_R"]
    maps = []
    ii = (np.arange(S) + 0.5) / S
    for b in range(B):
        cx, cy = rng.uniform(0.3, 0.7, 2)
        m = np.exp(-((ii[:, None] - cx) ** 2 + (ii[None, :] - cy) ** 2) / (2 * 0.03 ** 2))
        maps.append(m / m.sum())
    dm = torch.as_tensor(np.stack(maps), device=DEV)
    got = env.density_map_to_action(dm, agent_id=torch.zeros(B, dtype=torch.int32, device=DEV)).cpu().numpy()
    xy = np.stack([st["x"], st["y"]], 1)
    alive = env.view("status").cpu().numpy()
    counts = dict(exact=0, moved=0, close=0)
    reach = []
    for b in range(B):
        ref, res, x0, objective = _oracle_decode(env, None, b, maps[b])
        np.testing.assert_allclose(got[b, 2], ref[2], rtol=1e-12)
        reach.append(int(((np.hypot(*(xy - x0).T) <= R * 2.4143) & (alive[b] != 0)).sum()))
        loc = _locate_counts(env, got[b], ref, b, res, x0, counts)
        assert np.all(np.abs(loc - x0) <= R * (1 + 1e-12)), (b, loc, x0)
        assert -objective(loc) >= -objective(x0) * (1 - 1e-12), b
    print("dense field: %d to %d alive nodes within reach; %d decodes at scipy's box centre exactly, %d of %d others within 1e-3 m"
          % (min(reach), max(reach), counts["exact"], counts["close"], counts["moved"]))
    assert min(reach) > 64
    assert counts["close"] >= 0.9 * counts["moved"], counts
