"""Observation rasters (``wrsn_observe``: ``k_observe<double>``, ``k_observe<float>`` chunked, ``k_observe_win``) against the
float64 restatement of ``WRSN.get_state`` (oracle/obs_oracle.py), across map sizes, field shapes, node and charger counts.

The restatement is pinned first, against the golden episodes and against the C oracle.  Then every case builds a batch,
steps it, edits its state (dead node, node without traffic, chargers in the frame's corners and on its edges, both charger
types, a dead charger, padding nodes of a smaller scenario made alive), and compares the raster of every charger as the
observer with the restatement fed the state the simulator holds:
  float64 raster: 1e-12 of the channel maximum (same source order and roundings, only CUDA's exp differs, <= 1 ulp);
  float32 rasters: 1e-5 of the channel maximum.
At the map sizes and fields the windowed kernel accepts, the default path (windowed) and the chunked path (forced by
``dims.obs_sigma_cells = 0``) both run on the same state.  Every case checks that it is sensitive: dropping any one source,
or moving it by one cell, changes the restatement by more than twice the float32 bound.
The same harness runs on the host build (``-m "not gpu"``), whose ``wrsn_observe`` is the float64 restatement in C."""
import os
import subprocess

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import BatchedWRSN, Scenario, synthetic
from oracle import obs_oracle as oo
from oracle.wrsn_oracle import DEFAULT_MC, OracleWRSN, scenario_from_dict
from tests import helpers
from tests.helpers import REPO, golden, golden_names, mc_dict_of

EMU_DIR = os.path.join(REPO, "tests", "emu")
GPU = "cuda:0"
F64_BOUND = 1e-12
F32_BOUND = 1e-5
B = 4                                               # rows 0..2 observe, row 3 has agent_id -1
SENTINEL = -3.25


# ------------------------------------------------------------------ 1. the restatement itself
def _consts_of_golden(g):
    mc, sp = mc_dict_of(g), g["sc_par"]
    return dict(charging_range=mc["charging_range"], alpha=mc["alpha"], beta=mc["beta"], threshold=float(sp[1]),
                capacity=float(sp[0]), mc_capacity=mc["capacity"], velocity=mc["velocity"],
                charging_time_max=float(g["charging_time_max"]), moving_time_max=float(g["moving_time_max"]))


@pytest.mark.parametrize("name", golden_names("ep_"))
def test_reference_matches_golden_observations(name):
    """Every decision of every golden episode: channel sums and the stored full observations, at the tolerances of
    parity_cases.check_episode."""
    g = golden(name)
    S, consts = int(g["map_size"]), _consts_of_golden(g)
    full = {int(i): k for k, i in enumerate(g["full_state_idx"])}
    xy = np.asarray(g["sc_nodes"], np.float64).reshape(-1, 2)
    checked = 0
    for i in range(int(g["n"])):
        ag = int(g["agent_id"][i])
        if ag < 0:
            continue
        mc = np.column_stack([g["mc_loc"][i], g["mc_energy"][i], g["mc_cpa"][i], g["mc_type"][i]])
        st = oo.get_state(g["frame"], xy, g["status"][i], g["energy"][i], g["cs"][i], mc, ag, S, consts)
        np.testing.assert_allclose(st.reshape(4, -1).sum(1), g["chan_sum"][i], rtol=1e-9, atol=1e-9)
        if i in full:
            np.testing.assert_allclose(st, g["full_state"][full[i]], rtol=1e-9, atol=1e-12)
        checked += 1
    assert checked > 0


@pytest.mark.parametrize("S", [1, 7, 33, 100, 177])
def test_reference_matches_c_oracle(S):
    """orc_get_state (oracle/wrsn_oracle.c) of every charger at several decisions, within 1e-12 of the channel maximum."""
    sc = synthetic(num_nodes=100, num_targets=100, seed=11)
    o = OracleWRSN(scenario_from_dict(sc.to_dict()), num_agent=3, map_size=S)
    rng = np.random.default_rng(S)
    r = o.reset()
    checked = 0
    for _ in range(4):
        nd, m, c = o.nodes(), o.mcs(), o.consts()
        mc = np.column_stack([m["loc"], m["energy"], m["cpa"], m["type"]])
        consts = dict(charging_range=DEFAULT_MC["charging_range"], alpha=DEFAULT_MC["alpha"], beta=DEFAULT_MC["beta"],
                      threshold=float(o.sc["par"][1]), capacity=float(o.sc["par"][0]), mc_capacity=DEFAULT_MC["capacity"],
                      velocity=DEFAULT_MC["velocity"], charging_time_max=c["charging_time_max"], moving_time_max=c["moving_time_max"])
        for a in range(3):
            want = o.get_state(a)
            got = oo.get_state(c["frame"], o._nodes, nd["status"], nd["energy"], nd["cs"], mc, a, S, consts)
            for ch in range(4):
                assert np.abs(got[ch] - want[ch]).max() <= F64_BOUND * np.abs(want[ch]).max(), (S, a, ch)
            checked += 1
        act = rng.uniform(0, 1, 3); act[2] *= 0.05
        r = o.step(r["raw_agent_id"], act)
        if r["raw_agent_id"] < 0:
            break
    assert checked >= 6


# ------------------------------------------------------------------ 2. cases
def _scaled(sc, width, height=None):
    """``sc`` with nodes, targets and base station mapped affinely onto a field of width x height metres (the frame is
    their bounding box, Network.py:16-27)."""
    pts = np.vstack([sc.nodes, sc.base_station[None, :]])
    lo, hi = pts.min(0), pts.max(0)
    k = np.array([width, width if height is None else height]) / (hi - lo)
    f = lambda p: lo + (np.asarray(p, np.float64) - lo) * k
    return Scenario(nodes=f(sc.nodes), targets=f(sc.targets), base_station=f(sc.base_station),
                    node_phy_spe=dict(sc.node_phy_spe), max_time=sc.max_time)


def _field(kind, n):
    if kind == "square":                             # 1 km square at 100 nodes, the synthetic fields' density otherwise
        return [_scaled(synthetic(num_nodes=n, num_targets=100, seed=21), 1000.0 * np.sqrt(n / 100.0))]
    if kind == "rect":                               # 1000 x 1150 m: hx != hy, still narrow enough for the window
        return [_scaled(synthetic(num_nodes=132, num_targets=100, seed=22), 1000.0, 1150.0)]
    if kind == "strip":                              # 1000 x 300 m: 9 cells wide sources at S = 100, chunked
        return [_scaled(synthetic(num_nodes=100, num_targets=100, seed=23), 1000.0, 300.0)]
    if kind == "small":                              # synthetic(40): a 632 m field
        return [synthetic(num_nodes=40, num_targets=40, seed=24)]
    if kind == "sigma_in":                           # obs_sigma_cells = 27 / 932 * 100 = 2.897 at S = 100
        return [_scaled(synthetic(num_nodes=100, num_targets=100, seed=25), 932.0)]
    if kind == "sigma_out":                          # 27 / 930 * 100 = 2.903
        return [_scaled(synthetic(num_nodes=100, num_targets=100, seed=25), 930.0)]
    if kind == "mixed":                              # rows of 82 and 100 nodes: the 82-node rows carry 18 padding nodes
        return [_scaled(synthetic(num_nodes=82, num_targets=60, seed=26), 880.0),
                _scaled(synthetic(num_nodes=100, num_targets=100, seed=27), 1000.0)]
    raise KeyError(kind)


# (id, S, field, nodes, chargers, windowed-eligible at the default obs_sigma_cells)
CASES = ([("size%d" % S, S, "square", 100, 3, False) for S in (1, 2, 3, 7, 17, 32, 50, 64, 99, 101, 128, 176, 177, 256)]
         + [("win%d" % S, S, "square", 100, 3, True) for S in (40, 60, 80, 100)]
         + [("rect", 100, "rect", 132, 3, True), ("strip", 100, "strip", 100, 3, False),
            ("small100", 100, "small", 40, 3, False), ("small40", 40, "small", 40, 3, True),
            ("sigma_in", 100, "sigma_in", 100, 3, True), ("sigma_out", 100, "sigma_out", 100, 3, False),
            ("n500", 100, "square", 500, 3, False), ("m1", 100, "square", 100, 1, True), ("m16", 100, "square", 100, 16, True),
            ("mixed100", 100, "mixed", 100, 3, False), ("mixed60", 60, "mixed", 100, 3, True)])


def windowed_eligible(d):
    """wrsn_observe's choice of k_observe_win (wrsn_kernels.cu), restated: narrow sources, a map size the window's tiles
    cover, and the staged sources within 100 KB of shared memory."""
    sg = np.float32(d.obs_sigma_cells)
    wsmem = 4 * ((d.N + 2 * d.M) * (40 + 40 + 2 * 16) + 2 * d.obs_pitch) + 8 * (d.N + 2 * d.M)
    return bool(sg > 0 and sg <= np.float32(2.9) and d.S % 20 == 0 and d.S >= 40
                and (d.S // 4) * (d.S // 20) <= 128 and wsmem <= 100 * 1024)


def _set_state(env, S, rng):
    """The edits every case carries: node weights within ~30x of each other, one dead node, one node without traffic,
    padding nodes alive (they must still contribute nothing), chargers in the four corners with destinations on the
    frame's edges and at the window's tightest offset, both charger types, the last charger dead."""
    E = env.E
    status, energy, cs, mc = env.view("status"), env.view("energy"), env.view("cs"), env.view("mc")
    N, M = env.N, env.M
    nn = env.num_nodes.cpu().numpy()
    for b in range(env.B):
        par = env.statics[int(env.scen_id[b])]["par"]
        thr, cap = par["THR"], par["CAP"]
        f0, f1, f2, f3 = par["F0"], par["F1"], par["F2"], par["F3"]
        W, H = f1 - f0, f3 - f2
        e = thr + (cap - thr) * rng.uniform(0.3, 0.9, N)
        c = rng.uniform(0.01, 0.1, N)
        energy[b] = torch.as_tensor(e, dtype=energy.dtype)
        cs[b] = torch.as_tensor(c, dtype=cs.dtype)
        status[b] = 1                                 # includes the padding columns of a smaller scenario
        status[b, 3] = 0                              # a dead node
        cs[b, 5] = 0.0                                # a node without traffic: exact zeros, skipped by the kernels
        corners = [(f0, f2), (f1, f2), (f0, f3), (f1, f3)]
        for a in range(M):
            row = {}
            row["X"], row["Y"] = corners[a % 4]
            if S >= 7:
                kind = a % 4
                if kind == 0:                         # on the left edge
                    cx, cy = f0, f2 + H * rng.uniform(0.2, 0.8)
                elif kind == 1:                       # on the top edge
                    cx, cy = f0 + W * rng.uniform(0.2, 0.8), f3
                else:                                 # x0 * S just below 4k + 3: a 16.5-cell margin to the window's right end
                    k = int(rng.integers(0, max(1, (S - 3) // 4)))
                    cx = f0 + W * ((4 * k + 3 - 1e-6) / S)
                    cy = f2 + H * ((4 * int(rng.integers(0, max(1, (S - 3) // 4))) + 3 - 1e-6) / S) if kind == 3 else f2 + H * rng.uniform(0, 1)
            else:                                     # tiny maps: destinations at cell centres, where a 27 m source is visible
                cx = f0 + W * (int(rng.integers(0, S)) + 0.5) / S
                cy = f2 + H * (int(rng.integers(0, S)) + 0.5) / S
            row["CPA0"], row["CPA1"] = min(max(cx, f0), f1), min(max(cy, f2), f3)
            if a % 2 == 1:                            # a moving charger: far from its destination, travel times within 5x
                row["X"] = row["CPA0"] + (0.5 * W if row["CPA0"] < f0 + 0.5 * W else -0.5 * W)
            row["CPA2"] = rng.uniform(0.2, 0.8)
            row["ENERGY"] = par["MC_CAP"] * rng.uniform(0.3, 0.9)
            row["TYPE"] = float(a % 2 == 0)
            row["STATUS"] = 0.0 if (a == M - 1 and M > 1) else 1.0
            for k, v in row.items():
                mc[b, a, E["WRSN_MC_" + k]] = float(v)
        # a node source too narrow to show on a tiny map cannot be told from a missing one: those nodes are made dead
        if S < 17:
            srcs = _sources(env, b, 0, status, energy, cs, mc, nn)[0]
            terms = [(s[6], np.abs(oo.term(S, s, par["MTM"])).max()) for s in srcs]
            top = max([t for _, t in terms] + [0.0])
            for n, t in terms:
                if t < 1e-3 * top:
                    status[b, n] = 0


def _sources(env, b, observer, status, energy, cs, mc, nn):
    st = env.statics[int(env.scen_id[b])]
    par = st["par"]
    n = int(nn[b])
    E = env.E
    cols = [E["WRSN_MC_" + k] for k in ("X", "Y", "ENERGY", "CPA0", "CPA1", "CPA2", "TYPE")]
    mcr = mc[b, :env.M][:, cols].cpu().numpy()
    consts = dict(charging_range=par["MC_R"], alpha=par["MC_ALPHA"], beta=par["MC_BETA"], threshold=par["THR"],
                  capacity=par["CAP"], mc_capacity=par["MC_CAP"], velocity=par["MC_V"], charging_time_max=par["CTM"],
                  moving_time_max=par["MTM"])
    xy = np.stack([np.asarray(st["x"])[:n], np.asarray(st["y"])[:n]], 1)
    return oo.sources(st["frame"], xy, status[b, :n].cpu().numpy(), energy[b, :n].cpu().numpy(), cs[b, :n].cpu().numpy(),
                      mcr, observer, consts)


def _check_sensitive(S, srcs, ref, mtm, tag):
    """Dropping any one source, or moving it by one cell, must change the reference by more than twice the float32 bound."""
    for ch in range(4):
        live = [s for s in srcs[ch] if s[4] != 0.0]
        if not live:
            continue
        bound = 2 * F32_BOUND * np.abs(ref[ch]).max()
        for s in live:
            t = oo.term(S, s, mtm)
            step = -1.0 / S if s[0] < 0.5 else 1.0 / S         # away from the middle: never onto its mirror image
            moved = oo.term(S, (s[0] + step,) + tuple(s[1:]), mtm)
            assert np.abs(t).max() > bound, ("dropping a source is invisible", tag, ch, s[6])
            assert np.abs(moved - t).max() > bound, ("moving a source by one cell is invisible", tag, ch, s[6])


def run_case(case, device, on_gpu):
    """Build, step and edit one case; compare every raster path it selects with the reference.  Returns the largest error
    (relative to the channel maximum) per path."""
    cid, S, kind, n, M, eligible = case
    scs = _field(kind, n)
    env = BatchedWRSN(scs, num_agent=M, num_envs=B, map_size=S, device=device,
                      scenario_index=(np.arange(B) % 2) if kind == "mixed" else None)
    assert windowed_eligible(env.dims) == eligible, cid
    env.reset()
    g = torch.Generator(device="cpu"); g.manual_seed(S * 131 + M)
    for _ in range(3):
        a = torch.rand((B, 3), dtype=torch.float64, generator=g); a[:, 2] *= 0.05
        env.rollout_step(a.to(env.state.device))
    rng = np.random.default_rng(S * 7 + M)
    _set_state(env, S, rng)
    status, energy, cs, mc = env.view("status"), env.view("energy"), env.view("cs"), env.view("mc")
    nn = env.num_nodes.cpu().numpy()
    if kind == "mixed":
        assert nn.min() < env.N and status[nn.argmin(), int(nn.min()):].min() == 1     # alive padding nodes
    sigma = env.dims.obs_sigma_cells
    paths = [("fp64", torch.float64, sigma), ("fp32 chunked", torch.float32, 0.0)]
    if eligible:
        paths.append(("fp32 windowed", torch.float32, sigma))
    worst = {p[0]: 0.0 for p in paths}
    outs = {}
    for k in range(M):
        aid = torch.tensor([(b + k) % M for b in range(B - 1)] + [-1], dtype=torch.int32)
        refs = []
        for b in range(B - 1):
            srcs = _sources(env, b, int(aid[b]), status, energy, cs, mc, nn)
            mtm = env.statics[int(env.scen_id[b])]["par"]["MTM"]
            ref = oo.raster(S, srcs, mtm)
            _check_sensitive(S, srcs, ref, mtm, (cid, b, int(aid[b])))
            refs.append(ref)
        for name, dt, sg in paths:
            env.dims.obs_sigma_cells = sg
            out = torch.full((B, 4, S, S), SENTINEL, dtype=dt, device=env.state.device)
            env.get_state(agent_id=aid.to(env.state.device), out=out)
            got = out.cpu().numpy().astype(np.float64)
            outs[(name, k)] = out.cpu()
            assert np.all(got[B - 1] == SENTINEL), (cid, name)
            bound = F64_BOUND if dt == torch.float64 else F32_BOUND
            for b in range(B - 1):
                for ch in range(4):
                    mx = np.abs(refs[b][ch]).max()
                    err = np.abs(got[b, ch] - refs[b][ch]).max()
                    assert err <= bound * mx, (cid, name, k, b, ch, err / mx if mx else err)
                    if mx > 0:
                        worst[name] = max(worst[name], err / mx)
        env.dims.obs_sigma_cells = sigma
    print("%-10s S=%3d N=%3d M=%2d: largest error / channel maximum %s"
          % (cid, S, env.N, M, ", ".join("%s %.2e" % kv for kv in worst.items())))
    if on_gpu and eligible and S > 40:
        differ = any(not torch.equal(outs[("fp32 windowed", k)], outs[("fp32 chunked", k)]) for k in range(M))
        return worst, differ
    return worst, None


def test_case_matrix_covers_both_float32_paths():
    eligible = [c[5] for c in CASES]
    assert any(eligible) and not all(eligible)


# ------------------------------------------------------------------ 3. the harness on the host build
@pytest.fixture(scope="module")
def emu_built():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)


@pytest.fixture()
def host_build(emu_built):
    helpers.use_host_build()
    yield
    helpers.use_cuda_build_lazy()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_raster_harness_on_host_build(host_build, case):
    """The whole harness, state edits included, on the host build (its wrsn_observe is the float64 restatement; it ignores
    obs_sigma_cells, so every float32 path there is the float64 map rounded once)."""
    run_case(case, "cpu", on_gpu=False)


# ------------------------------------------------------------------ 4. the CUDA rasters
@pytest.fixture()
def cuda_library():
    L = helpers.use_cuda_build()
    assert not helpers.is_host_build(L) and torch.cuda.is_available()
    yield


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_raster_matches_reference(cuda_library, case):
    worst, differ = run_case(case, GPU, on_gpu=True)
    if differ is not None:
        # the forced path really ran: the windowed and the chunked float32 rasters of the same state differ in bits (at S = 40
        # the window spans the whole map and both kernels run the same FFMAs in the same order: equal bits are expected there)
        assert differ, case[0]
