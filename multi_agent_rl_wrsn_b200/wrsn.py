"""``WRSN`` — single-environment façade with the reference's constructor, request dict and attributes.

Drop-in for ``rl_env.WRSN.WRSN`` (``rl_env/WRSN.py:21-330``) as the controllers use it
(``controller/ippo/IPPO.py:137-183``, ``controller/random/RandomController.py:12``): ``reset()``,
``step(agent_id, input_action)``, ``num_agent``, ``env.now``, ``net.targets_active``, ``observation_space``,
``action_space``.  The simulation itself runs in the sm_100a kernels of ``BatchedWRSN`` with one environment;
use ``BatchedWRSN`` directly for throughput.

A density-map action (``density_map=True``, the runners' setting) is decoded ON THE DEVICE (``wrsn_decode_density_map``:
see DESIGN §4.4 for what is reproduced exactly); there is no host-side decode in this package.  The views in ``info`` read
from ONE host copy of the environment's record per request (a single device-to-host transfer), not from one transfer per
attribute.

Differences from the reference, on purpose:
  * the request carries ``detailed_rewards`` = [term_all, term_exclusive, reward]; the reference's controllers read that
    key (``IPPO.py:162-164``) although its environment never writes it (SURVEY Q10);
  * ``info`` holds light read-only views (``net``, ``agents``) backed by device state instead of live SimPy objects;
  * if every charger is dead the reference's ``step`` never returns (Q1); here it raises ``RuntimeError``.
"""
import numpy as np
import torch
import yaml

from .batched import BatchedWRSN
from .scenario import Scenario


class Box:
    """Minimal ``gym.spaces.Box`` stand-in (``low`` / ``high`` / ``shape`` / ``dtype``), WRSN.py:31-32."""

    def __init__(self, low, high, shape, dtype):
        self.low = np.full(shape, low, dtype)
        self.high = np.full(shape, high, dtype)
        self.shape, self.dtype = tuple(shape), dtype

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)


class _Clock:
    def __init__(self, owner):
        self._o = owner

    @property
    def now(self):
        return float(self._o._host("hdr")[self._o._b.E["WRSN_H_NOW"]])


class _NodeView:
    def __init__(self, net, i):
        self._n, self.id = net, i

    @property
    def location(self):
        return self._n._xy[self.id]

    @property
    def energy(self):
        return float(self._n._o._host("energy")[self.id])

    @property
    def energyCS(self):
        return float(self._n._o._host("cs")[self.id])

    @property
    def energyRR(self):
        return float(self._n._o._host("rr")[self.id])

    @property
    def status(self):
        return int(self._n._o._host("status")[self.id])

    @property
    def level(self):
        return int(self._n._o._host("level")[self.id])


class _NetView:
    def __init__(self, owner):
        self._o = owner
        sc = owner._b.scenarios[0]
        st = owner._b.statics[0]
        self._xy = np.array(sc.nodes, np.float64)
        self.frame = np.array(st["frame"], np.float64)
        self.nodes_density = st["nodes_density"]
        self.listNodes = [_NodeView(self, i) for i in range(sc.N)]
        self.listTargets = [np.array(t, np.float64) for t in sc.targets]
        self.baseStation = type("BaseStationView", (), {"location": np.array(sc.base_station, np.float64)})()
        self.max_time = sc.max_time
        self.env = owner.env

    @property
    def targets_active(self):
        w = self._o._host("tact_words").astype(np.int64) & 0xFFFFFFFF
        bits = (w[:, None] >> np.arange(32)) & 1
        return [int(v) for v in bits.reshape(-1)[:self._o._b.T]]

    @property
    def alive(self):
        return int(self._o._host("hdr")[self._o._b.E["WRSN_H_ALIVE"]])


class _AgentView:
    def __init__(self, owner, i):
        self._o, self.id = owner, i
        mc = owner._b.mc_type
        self.capacity, self.threshold = mc["capacity"], mc["threshold"]
        self.alpha, self.beta, self.velocity, self.pm = mc["alpha"], mc["beta"], mc["velocity"], mc["pm"]
        self.chargingRange, self.epsilon = mc["charging_range"], mc["epsilon"]

    def _f(self, name):
        return float(self._o._host("mc")[self.id, self._o._b.E["WRSN_MC_" + name]])

    @property
    def location(self):
        return np.array([self._f("X"), self._f("Y")])

    @property
    def energy(self):
        return self._f("ENERGY")

    @property
    def status(self):
        return int(self._f("STATUS"))

    @property
    def cur_phy_action(self):
        return [self._f("CPA0"), self._f("CPA1"), self._f("CPA2")]

    @property
    def cur_action_type(self):
        return "charging" if self._f("TYPE") != 0.0 else "moving"


class WRSN:
    def __init__(self, scenario_path, agent_type_path, num_agent, map_size=100, warm_up_time=100, density_map=False,
                 device=None):
        """Same arguments as the reference's constructor (``rl_env/WRSN.py:22``), plus the CUDA device."""
        scenario = scenario_path if isinstance(scenario_path, Scenario) else Scenario.load_yaml(scenario_path)
        if isinstance(agent_type_path, dict) or agent_type_path is None:
            self.agent_phy_para = agent_type_path
        else:
            with open(agent_type_path) as f:
                self.agent_phy_para = yaml.safe_load(f)
        self.num_agent, self.map_size = int(num_agent), int(map_size)
        self.density_map, self.warm_up_time = bool(density_map), warm_up_time
        self.epsilon = 1e-9
        self.observation_space = Box(0.0, 1.0, (4, self.map_size, self.map_size), np.float64)
        self.action_space = Box(0.0, 1.0, (3,), np.float64)
        self._b = BatchedWRSN(scenario, num_agent=self.num_agent, mc_type=self.agent_phy_para, num_envs=1,
                              map_size=self.map_size, warm_up_time=warm_up_time, device=device)
        self.agent_phy_para = self._b.mc_type
        par = self._b.statics[0]["par"]
        self.moving_time_max, self.charging_time_max, self.avg_nodes_agent = par["MTM"], par["CTM"], par["AVGNA"]
        self.env = _Clock(self)
        self.net = _NetView(self)
        self.agents = [_AgentView(self, i) for i in range(self.num_agent)]
        self.agents_input_action = [None] * self.num_agent
        self.agents_prev_state = [None] * self.num_agent
        self._row = None
        self.reset()

    # ------------------------------------------------------------------ reference helpers (WRSN.py:86-98)
    def down_mapping(self, location):
        f = self.net.frame
        return np.array([(location[0] - f[0]) / (f[1] - f[0]), (location[1] - f[2]) / (f[3] - f[2])])

    def up_mapping(self, down_map):
        f = self.net.frame
        return np.array([down_map[0] * (f[1] - f[0]) + f[0], down_map[1] * (f[3] - f[2]) + f[2]])

    def translate(self, agent_id, action):
        f = self.net.frame
        return np.array([action[0] * (f[1] - f[0]) + f[0], action[1] * (f[3] - f[2]) + f[2], self.charging_time_max * action[2]])

    def get_state(self, agent_id):
        a = torch.full((1,), int(agent_id), dtype=torch.int32, device=self._b.device)
        return self._b.get_state(agent_id=a, dtype=torch.float64)[0].cpu().numpy()

    def get_network_fitness(self):
        return self._b.get_network_fitness()[0][0].cpu().numpy()

    # ------------------------------------------------------------------ WRSN.density_map_to_action (:229-287)
    def density_map_to_action(self, dmap, id):
        """An S x S density map (already a distribution, as ``WRSN.step`` hands it over, or raw: the device applies the same
        normalisation rule, ``:293-296``) -> the 3-vector action, decoded by ``wrsn_decode_density_map`` on the device."""
        dm = torch.as_tensor(np.ascontiguousarray(dmap, np.float64).reshape(1, self.map_size, self.map_size), device=self._b.device)
        aid = torch.tensor([int(id)], dtype=torch.int32, device=self._b.device)
        return self._b.density_map_to_action(dm, agent_id=aid)[0].cpu().numpy()

    def heuristic_action(self, agent_id, kind="min_lifetime"):
        """The hand-written charging decision of charger ``agent_id`` (``BatchedWRSN.heuristic_action``) -> the 3-vector
        action, for ``step`` of an environment built with ``density_map=False``."""
        aid = torch.tensor([int(agent_id)], dtype=torch.int32, device=self._b.device)
        return self._b.heuristic_action(kind, agent_id=aid)[0].cpu().numpy()

    def _host(self, name):
        """Typed view of ONE host copy of the environment's record, fetched once per request (invalidated by reset / step)."""
        if self._row is None:
            self._row = self._b.state.cpu()
        return self._b.view(name, self._row)[0].numpy()

    # ------------------------------------------------------------------ reset / step
    def _request(self, req, agent_in=None):
        self._row = None                                 # the views refetch the record when they are next read
        pack = torch.cat([req.agent_id.to(torch.float64), req.flags.to(torch.float64), req.terminal.to(torch.float64),
                          req.reward, req.detail.reshape(-1), req.action.reshape(-1)]).cpu().numpy()   # one transfer
        aid, flags, terminal, reward, det, action = int(pack[0]), int(pack[1]), bool(pack[2]), float(pack[3]), pack[4:6], pack[6:9]
        if flags & 2:
            raise RuntimeError("wrsn_b200 engine error %g" % float(self._host("hdr")[self._b.E["WRSN_H_ERR"]]))
        if flags & 1:
            raise RuntimeError("every mobile charger is dead: the reference's WRSN.step would never return (SURVEY Q1)")
        info = [self.net, self.agents]
        if aid == -2:                                # the reference falls off the end of step() and returns None (Q7)
            return None
        if aid < 0:
            return {"agent_id": None, "prev_state": None, "input_action": None, "action": None, "reward": None,
                    "state": None, "terminal": terminal, "info": info, "detailed_rewards": None}
        state = self.get_state(aid)
        prev = self.agents_prev_state[aid] if self.agents_prev_state[aid] is not None else state
        return {"agent_id": aid, "prev_state": prev, "input_action": self.agents_input_action[aid],
                "action": action.copy(), "reward": reward, "state": state, "terminal": terminal,
                "info": info, "detailed_rewards": [float(det[0]), float(det[1]), reward]}

    def reset(self):
        req = self._b.reset()
        self.agents_input_action = [None] * self.num_agent
        self.agents_prev_state = [None] * self.num_agent
        out = self._request(req)
        if out is not None and out["agent_id"] is not None:
            self._last_state = (out["agent_id"], out["state"])
        return out

    def step(self, agent_id, input_action):
        dev = self._b.device
        if agent_id is not None:
            action = np.array(input_action)
            self.agents_input_action[agent_id] = action.copy()
            if self.density_map:                         # normalisation (:293-296) + decode (:229-287) on the device
                action = self.density_map_to_action(action, agent_id)
            # prev_state = get_state(agent_id) before the simulation advances == the state last handed out for it
            last = getattr(self, "_last_state", None)
            self.agents_prev_state[agent_id] = last[1] if last is not None and last[0] == agent_id else self.get_state(agent_id)
            a = torch.tensor([agent_id], dtype=torch.int32, device=dev)
            x = torch.as_tensor(np.asarray(action, np.float64).reshape(1, 3), device=dev)
        else:
            a = torch.tensor([-1], dtype=torch.int32, device=dev)
            x = torch.zeros((1, 3), dtype=torch.float64, device=dev)
        out = self._request(self._b.step(a, x))
        if out is not None and out["agent_id"] is not None:
            self._last_state = (out["agent_id"], out["state"])
        return out
