"""ctypes binding of the C restatement ``oracle/wrsn_oracle.c`` (TEST INFRASTRUCTURE).

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import yaml

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

DEFAULT_MC = dict(capacity=108000, threshold=0, velocity=5, pm=1, charging_range=27, alpha=4500, beta=30,
                  epsilon=1e-10)      # physical_env/mc/mc_types/default.yaml:2-9


def build(force=False):
    so = os.path.join(_HERE, "libwrsn_oracle.so")
    src = os.path.join(_HERE, "wrsn_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libwrsn_oracle.so"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.orc_create.restype = C.c_void_p
        L.orc_create.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, C.c_int, dp, C.c_int, C.c_double]
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_start_network_only.argtypes = [C.c_void_p]
        L.orc_run_until.argtypes = [C.c_void_p, C.c_double]
        L.orc_netop_done.argtypes = [C.c_void_p]
        L.orc_netop_done.restype = C.c_int
        L.orc_get_state.argtypes = [C.c_void_p, C.c_int, dp]
        L.orc_fitness.argtypes = [C.c_void_p, dp]
        L.orc_fitness.restype = C.c_double
        L.orc_reset.argtypes = [C.c_void_p, dp, dp]
        L.orc_step.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp]
        L.orc_now.argtypes = [C.c_void_p]
        L.orc_now.restype = C.c_double
        L.orc_alive.argtypes = [C.c_void_p]
        L.orc_alive.restype = C.c_int
        L.orc_set_event_budget.argtypes = [C.c_void_p, C.c_longlong]
        L.orc_nevents.argtypes = [C.c_void_p]
        L.orc_nevents.restype = C.c_longlong
        L.orc_get_nodes.argtypes = [C.c_void_p, dp, dp, dp, dp, ip, ip]
        L.orc_get_targets_active.argtypes = [C.c_void_p, C.POINTER(C.c_ubyte)]
        L.orc_get_mc.argtypes = [C.c_void_p, dp]
        L.orc_get_consts.argtypes = [C.c_void_p, dp]
        L.orc_get_static.argtypes = [C.c_void_p, ip, ip, ip, ip, ip]
        L.orc_get_static.restype = C.c_int
        L.orc_set_node_energy.argtypes = [C.c_void_p, C.c_int, C.c_double]
        L.orc_set_mc_energy.argtypes = [C.c_void_p, C.c_int, C.c_double]
        _LIB = L
    return _LIB


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def load_scenario_yaml(path):
    """Reference schema (network_scenarios/*.yaml: node_phy_spe, seed, max_time, base_station, nodes, targets)."""
    with open(path) as f:
        d = yaml.safe_load(f)
    return scenario_from_dict(d)


def scenario_from_dict(d):
    spe = d["node_phy_spe"]
    par = np.array([spe["capacity"], spe["threshold"], spe["com_range"], spe["sen_range"], spe["prob_gp"],
                    spe["package_size"], spe["er"], spe["et"], spe["efs"], spe["emp"],
                    d.get("max_time", 604800)], np.float64)
    return dict(nodes=np.array(d["nodes"], np.float64).reshape(-1, 2),
                targets=np.array(d["targets"], np.float64).reshape(-1, 2),
                bs=np.array(d["base_station"], np.float64), par=par)


def mc_params(d=None):
    d = dict(DEFAULT_MC) if d is None else d
    return np.array([d["capacity"], d["threshold"], d["velocity"], d["pm"], d["charging_range"], d["alpha"],
                     d["beta"], d["epsilon"]], np.float64)


class OracleWRSN:
    """C-oracle twin of ``rl_env.WRSN.WRSN`` (reset/step with 3-vector actions) plus state accessors."""

    def __init__(self, scenario, num_agent=3, mc=None, map_size=100, warm_up_time=100.0):
        if isinstance(scenario, str):
            scenario = load_scenario_yaml(scenario)
        if isinstance(mc, str):
            with open(mc) as f:
                mc = yaml.safe_load(f)
        self.sc = scenario
        self.N, self.T, self.M, self.S = len(scenario["nodes"]), len(scenario["targets"]), num_agent, map_size
        self._nodes = np.ascontiguousarray(scenario["nodes"], np.float64)
        self._targets = np.ascontiguousarray(scenario["targets"], np.float64)
        self._bs = np.ascontiguousarray(scenario["bs"], np.float64)
        self._par = np.ascontiguousarray(scenario["par"], np.float64)
        self._mcp = mc_params(mc)
        self.L = lib()
        self.h = self.L.orc_create(self.N, self.T, _dp(self._nodes), _dp(self._targets), _dp(self._bs),
                                   _dp(self._par), self.M, _dp(self._mcp), self.S, float(warm_up_time))
        if not self.h:
            raise RuntimeError("orc_create failed")

    def __del__(self):
        try:
            if self.h:
                self.L.orc_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- pure network ------------------------------------------------------------
    def start_network_only(self):
        self.L.orc_start_network_only(self.h)

    def run_until(self, t):
        self.L.orc_run_until(self.h, float(t))

    def netop_done(self):
        return bool(self.L.orc_netop_done(self.h))

    # -- WRSN API -------------------------------------------------------------------
    def _req(self, r, state, prev_state=None):
        aid = int(r[0])
        return dict(agent_id=None if aid < 0 else aid, raw_agent_id=aid, terminal=bool(r[1]), reward=float(r[2]),
                    action=r[3:6].copy(), now=float(r[6]), hang=bool(r[7]),
                    state=state if aid >= 0 else None, prev_state=prev_state if aid >= 0 else None)

    def reset(self, want_state=True):
        r = np.zeros(8)
        st = np.zeros((4, self.S, self.S)) if want_state else None
        self.L.orc_reset(self.h, _dp(r), _dp(st) if want_state else None)
        return self._req(r, st, st)

    def step(self, agent_id, action, want_state=True, want_prev=False):
        r = np.zeros(8)
        st = np.zeros((4, self.S, self.S)) if want_state else None
        pst = np.zeros((4, self.S, self.S)) if want_prev else None
        a = np.ascontiguousarray(action if action is not None else [0, 0, 0], np.float64)
        self.L.orc_step(self.h, -1 if agent_id is None else int(agent_id), _dp(a), _dp(r),
                        _dp(st) if want_state else None, _dp(pst) if want_prev else None)
        return self._req(r, st, pst)

    def set_event_budget(self, n):
        self.L.orc_set_event_budget(self.h, int(n))

    def set_node_energy(self, i, e):
        """TEST INFRASTRUCTURE: overwrite node i's energy (no event, no status check)."""
        self.L.orc_set_node_energy(self.h, int(i), float(e))

    def set_mc_energy(self, a, e):
        """TEST INFRASTRUCTURE: overwrite charger a's energy (no event)."""
        self.L.orc_set_mc_energy(self.h, int(a), float(e))

    # -- accessors --------------------------------------------------------------------
    @property
    def now(self):
        return self.L.orc_now(self.h)

    @property
    def alive(self):
        return self.L.orc_alive(self.h)

    def nodes(self):
        e, cs, rr, le = (np.zeros(self.N) for _ in range(4))
        st, lv = np.zeros(self.N, np.int32), np.zeros(self.N, np.int32)
        self.L.orc_get_nodes(self.h, _dp(e), _dp(cs), _dp(rr), _dp(le), _ip(st), _ip(lv))
        return dict(energy=e, cs=cs, rr=rr, log_energy=le, status=st.astype(np.uint8), level=lv)

    def targets_active(self):
        out = np.zeros(max(self.T, 1), np.uint8)
        self.L.orc_get_targets_active(self.h, out.ctypes.data_as(C.POINTER(C.c_ubyte)))
        return out[:self.T]

    def mcs(self):
        out = np.zeros((max(self.M, 1), 10))
        self.L.orc_get_mc(self.h, _dp(out))
        out = out[:self.M]
        return dict(loc=out[:, 0:2].copy(), energy=out[:, 2].copy(), status=out[:, 3].astype(np.uint8),
                    cpa=out[:, 4:7].copy(), type=out[:, 7].astype(np.uint8), nconn=out[:, 8].astype(np.int32),
                    excl=out[:, 9].copy())

    def consts(self):
        out = np.zeros(8)
        self.L.orc_get_consts(self.h, _dp(out))
        return dict(frame=out[:4].copy(), moving_time_max=out[4], charging_time_max=out[5],
                    avg_nodes_agent=out[6], nodes_density=out[7])

    def fitness(self):
        out = np.zeros(max(self.T, 1))
        mn = self.L.orc_fitness(self.h, _dp(out))
        return mn, out[:self.T]

    def get_state(self, agent_id):
        st = np.zeros((4, self.S, self.S))
        self.L.orc_get_state(self.h, int(agent_id), _dp(st))
        return st

    def static_graph(self):
        nbr_ptr = np.zeros(self.N + 1, np.int32)
        tgt_ptr = np.zeros(self.N + 1, np.int32)
        direct = np.zeros(self.N, np.int32)
        ne = self.L.orc_get_static(self.h, _ip(nbr_ptr), None, _ip(tgt_ptr), None, _ip(direct))
        nbr_idx = np.zeros(max(ne, 1), np.int32)
        tgt_idx = np.zeros(max(int(tgt_ptr[-1]), 1), np.int32)
        self.L.orc_get_static(self.h, _ip(nbr_ptr), _ip(nbr_idx), _ip(tgt_ptr), _ip(tgt_idx), _ip(direct))
        return dict(nbr_ptr=nbr_ptr, nbr_idx=nbr_idx[:ne], tgt_ptr=tgt_ptr, tgt_idx=tgt_idx[:tgt_ptr[-1]],
                    direct=direct)


def charge_rates_reference(nodes, status, mc_xy, charging, charging_range, alpha, beta):
    """TEST INFRASTRUCTURE.  The reference's charging model written out with its own statements: for every charger m
    (``charging[m]``) the ``connected_nodes`` of ``MobileCharger.charge`` (``physical_env/mc/MobileCharger.py:56-59``:
    ``euclidean(node.location, self.location) <= self.chargingRange``, nodes in list order) each run
    ``Node.charger_connection`` (``physical_env/network/Node.py:134-139``: nothing for a dead node, else
    ``tmp = mc.alpha / (euclidean(...) + mc.beta) ** 2; self.energyRR += tmp; mc.chargingRate += tmp``).
    Returns (energyRR per node, chargingRate per charger) as float64 arrays."""
    import math
    import numpy as np
    nodes = np.asarray(nodes, np.float64)
    rr = np.zeros(len(nodes), np.float64)
    cr = np.zeros(len(mc_xy), np.float64)
    for m, loc in enumerate(np.asarray(mc_xy, np.float64)):
        if not charging[m]:
            continue
        for n in range(len(nodes)):
            # scipy.spatial.distance.euclidean for 2-vectors = sqrt(dot(u, u)); written with Python floats so that the two
            # products and the sum are rounded separately on every host (a BLAS dot may fuse them: last-ulp, host-dependent,
            # SURVEY 8c) — the form the engine and the C oracle use
            ux, uy = float(nodes[n][0]) - float(loc[0]), float(nodes[n][1]) - float(loc[1])
            d = math.sqrt(ux * ux + uy * uy)
            if not d <= charging_range:
                continue
            if status[n] == 0:
                continue
            t = d + beta
            tmp = alpha / (t * t)                     # DESIGN §5: (d + beta) ** 2 as a product (libm pow differs by 1 ulp in 0.085 %)
            rr[n] += tmp
            cr[m] += tmp
    return rr, cr
