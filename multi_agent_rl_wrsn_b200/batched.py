"""``BatchedWRSN`` — B independent WRSN environments advanced in lockstep on one B200.

Host-side mirror of ``rl_env.WRSN.WRSN`` (``rl_env/WRSN.py:21``): the same ``reset`` / ``step`` /
``get_state`` / ``get_network_fitness`` contract, but every argument and result carries a leading
environment axis and lives in HBM as a torch tensor.  All simulation work happens in the sm_100a kernels
behind the C ABI of ``include/wrsn_b200.h``; torch is the allocator and the stream provider only.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .scenario import Scenario, build_static, load_mc_type
from .snapshot import LAYOUT_DIMS, REQ_FIELDS, EnvSnapshot, c_request, check_layout, layout_meta, scenario_fingerprint

_NP = {"f64": np.float64, "i32": np.int32, "u8": np.uint8}
HEURISTICS = ("min_lifetime", "nearest_urgent")     # wrsn_heuristic_action's kinds, in enum order (WRSN_HEUR_*)
_S_FIELDS = (  # (enum, dtype, which size)
    ("WRSN_S_PAR", "f64", "P"), ("WRSN_S_NX", "f64", "Npad"), ("WRSN_S_NY", "f64", "Npad"),
    ("WRSN_S_BS_ESEND", "f64", "Npad"), ("WRSN_S_NBR_DIST", "f64", "Emax"), ("WRSN_S_NBR_ESEND", "f64", "Emax"),
    ("WRSN_S_NBR_PTR", "i32", "Npad1"), ("WRSN_S_TGT_PTR", "i32", "Npad1"), ("WRSN_S_NBR_IDX", "i32", "Emax"),
    ("WRSN_S_TGT_IDX", "i32", "TEmax"), ("WRSN_S_DIRECT", "u8", "Npad"))


class Requests:
    """The request record of ``WRSN.reset`` / ``WRSN.step`` (``WRSN.py:68-83,313-330``) for every environment.

    ``agent_id``: >= 0 deciding charger, -1 ``None`` (terminal), -2 implicit ``None`` (SURVEY Q7), -3 row not
    touched by the call (masked out), -4 the step is still in flight (``step_budget`` exhausted: the next ``step`` /
    ``rollout_step`` continues it, whatever agent / action it is handed for that row).  ``flags`` bit0: every charger is
    dead (the reference would never return, Q1); bit1: engine error.
    """

    def __init__(self, B, device):
        self.agent_id = torch.full((B,), -3, dtype=torch.int32, device=device)
        self.terminal = torch.zeros((B,), dtype=torch.uint8, device=device)
        self.reward = torch.zeros((B,), dtype=torch.float64, device=device)
        self.now = torch.zeros((B,), dtype=torch.float64, device=device)
        self.action = torch.zeros((B, 3), dtype=torch.float64, device=device)
        self.detail = torch.zeros((B, 2), dtype=torch.float64, device=device)
        self.flags = torch.zeros((B,), dtype=torch.int32, device=device)
        self.stats = torch.zeros((B, 3), dtype=torch.float64, device=device)   # running totals: decisions, simulated seconds, resets
        self.sticky = torch.zeros((B,), dtype=torch.int32, device=device)      # OR of every `flags` value written so far (see raise_on_error)
        self.order = torch.zeros((B,), dtype=torch.int32, device=device)       # scratch: launch order of the step kernel's CTAs (longest step first)
        self.c = _lib.Request(self.agent_id.data_ptr(), self.terminal.data_ptr(), self.reward.data_ptr(),
                              self.now.data_ptr(), self.action.data_ptr(), self.detail.data_ptr(), self.flags.data_ptr(),
                              self.stats.data_ptr(), self.sticky.data_ptr(), self.order.data_ptr())


def episode_ends(req, running, decisions, cap):
    """Which of the rows ``running`` end their episode at the request ``req`` (``controllers.evaluate``'s rule): -> (terminal,
    ended).  Terminal: the request names no charger (``agent_id == -1``).  Ended: terminal, or (``cap`` not None) a request
    that is not in flight after ``cap`` decisions."""
    terminal = running & (req.agent_id == -1)
    ended = terminal
    if cap is not None:
        ended = ended | (running & (req.agent_id != -1) & (req.agent_id != -4) & (decisions >= cap))
    return terminal, ended


def episode_step(env, running, action, decisions, returns):
    """One ``step`` of the rows ``running`` of ``env`` and ``controllers.evaluate``'s accounting of it: a request with no deciding
    charger (-2) is stepped with agent -1, a step in flight (-4) continues; ``decisions`` counts the actions handed to a deciding
    charger, ``returns`` adds the reward of the next request (NaN counted as 0)."""
    aid = env.req.agent_id
    decided = running & (aid >= 0)
    env.step(torch.where(aid >= 0, aid, torch.full_like(aid, -1)), action, mask=running)
    decisions += decided.to(torch.int64)
    returns += torch.where(running, torch.nan_to_num(env.req.reward, nan=0.0), torch.zeros_like(returns))


class BatchedWRSN:
    def __init__(self, scenarios, num_agent=3, mc_type=None, num_envs=None, scenario_index=None, map_size=100,
                 warm_up_time=100, device=None, threads=0, step_budget=0, step_rounds=0):
        """``scenarios``: one or several ``Scenario`` / YAML paths, possibly of different sizes;
        ``scenario_index[b]`` picks the scenario of environment b (default: round robin).  Every environment simulates
        exactly its own scenario.  ``self.N`` / ``self.T`` are the largest node and target counts of the batch and
        ``self.num_nodes`` / ``self.num_targets`` (int32 [B] on the device) each row's own.  Per-node and per-target views
        keep the shape [B, N] / [B, T]: the columns beyond a row's own count are padding (status 0, energy 0,
        ``targets_active`` 0, fitness 0, never written by the kernels).  All rows run on the thread count of the largest
        scenario.  ``num_agent``, ``mc_type``, ``map_size`` and ``warm_up_time`` are the same for the whole batch.
        ``step_budget`` (``wrsn_dims.step_budget``, may be changed later through ``self.dims``): 0 = every ``step`` returns
        the environment's next request, as the reference does; > 0 = work units per launch and environment — a step that
        needs more comes back with ``agent_id == -4`` and continues at the next call, so one launch over thousands of
        environments lasts as long as the budget instead of as long as its slowest environment.
        ``step_rounds`` (``wrsn_dims.step_rounds``, with a budget): R > 0 cuts a step by kind of work as well — R rounds of
        two launches per call, the events kernel and the batch kernel that holds nothing but the hot second-by-second
        loop (same results, better instruction-cache behaviour; see include/wrsn_b200.h).  R < 0 is rejected."""
        self.L = _lib.lib()
        self.device = self._require_device(device)
        if isinstance(scenarios, (str, Scenario)):
            scenarios = [scenarios]
        self.scenarios = [s if isinstance(s, Scenario) else Scenario.load_yaml(s) for s in scenarios]
        self.mc_type = load_mc_type(mc_type)
        self.num_agent = int(num_agent)
        self.map_size = int(map_size)
        self.warm_up_time = float(warm_up_time)
        statics = [build_static(s, self.mc_type, self.warm_up_time) for s in self.scenarios]
        self.statics = statics
        N, T = max(st["N"] for st in statics), max(st["T"] for st in statics)
        n_scen = len(statics)
        B = int(num_envs) if num_envs is not None else (len(scenario_index) if scenario_index is not None else n_scen)
        self.B, self.N, self.T, self.M, self.S = B, N, T, self.num_agent, self.map_size
        self.E = _lib.enums()
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S = B, N, T, self.M, self.S
        d.Emax = max(len(st["nbr_idx"]) for st in statics)
        d.TEmax = max(len(st["tgt_idx"]) for st in statics)
        d.n_scen, d.threads = n_scen, int(threads)
        self._call(self.L.wrsn_dims_finalize, C.byref(d))
        d.step_budget, d.step_rounds = int(step_budget), int(step_rounds)
        # widest node / charger source of get_state in map cells: narrow sources take the windowed float32 raster
        d.obs_sigma_cells = max(float(self.mc_type["charging_range"]) / min(st["frame"][1] - st["frame"][0], st["frame"][3] - st["frame"][2])
                                for st in statics) * self.S
        self.dims = d
        self._foff = (C.c_int64 * self.E["WRSN_F_COUNT"])()
        self._soff = (C.c_int64 * self.E["WRSN_S_COUNT"])()
        self._call(self.L.wrsn_state_layout, C.byref(d), self._foff)
        self._call(self.L.wrsn_scen_layout, C.byref(d), self._soff)

        self.scen = torch.from_numpy(self._pack_scenarios(statics)).to(self.device)
        self._call(self.L.wrsn_build_obs_tables, C.byref(d), self.scen.data_ptr(), self._stream())
        if scenario_index is None:
            scenario_index = np.arange(B) % n_scen
        self.scen_id = torch.as_tensor(np.asarray(scenario_index, np.int32), device=self.device)
        sid = np.asarray(scenario_index, np.int64)
        self.num_nodes = torch.as_tensor(np.array([statics[k]["N"] for k in sid], np.int32), device=self.device)
        self.num_targets = torch.as_tensor(np.array([statics[k]["T"] for k in sid], np.int32), device=self.device)
        self.state = torch.zeros((B, d.state_bytes), dtype=torch.uint8, device=self.device)
        self.req = Requests(B, self.device)
        self._all = None
        self._snap = None
        self._agent_obs = None
        self._fingerprints = None
        self._counts = None
        self._branches = {}                              # lookahead's branch batches, one per width
        self._make_snapshot()

    # ------------------------------------------------------------------ plumbing
    def _require_device(self, device):
        """The sm_100 device this simulator lives on.  There is no CPU path: anything else raises."""
        dev = torch.device("cuda" if device is None else device)
        if dev.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("BatchedWRSN needs a CUDA device (sm_100a); there is no CPU path")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(dev):
            if not self.L.wrsn_device_ok():
                raise RuntimeError("wrsn_b200: " + self.L.wrsn_last_error().decode())
        return dev

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _sync(self):
        torch.cuda.synchronize(self.device)

    def _call(self, fn, *args):
        """Every launch runs with THIS simulator's device current (the C ABI launches on the CUDA runtime's current device;
        the stream handle alone does not select it)."""
        if torch.cuda.current_device() != self.device.index:
            with torch.cuda.device(self.device):
                rc = fn(*args)
        else:
            rc = fn(*args)
        _lib.check(rc, self.L)

    def _pack_scenarios(self, statics):
        d, E = self.dims, self.E
        buf = np.zeros((d.n_scen, d.scen_bytes), np.uint8)
        sizes = dict(P=E["WRSN_P_LEN"], Npad=d.Npad, Npad1=d.Npad + 1, Emax=d.Emax, TEmax=d.TEmax)
        for s, st in enumerate(statics):
            par = np.zeros(E["WRSN_P_LEN"], np.float64)
            for k, v in st["par"].items():
                par[E["WRSN_P_" + k]] = v
            n = st["N"]
            ptr_n = np.full(d.Npad + 1, st["nbr_ptr"][-1], np.int32); ptr_n[:n + 1] = st["nbr_ptr"]
            ptr_t = np.full(d.Npad + 1, st["tgt_ptr"][-1], np.int32); ptr_t[:n + 1] = st["tgt_ptr"]
            vals = dict(WRSN_S_PAR=par, WRSN_S_NX=st["x"], WRSN_S_NY=st["y"], WRSN_S_BS_ESEND=st["bs_esend"],
                        WRSN_S_NBR_DIST=st["nbr_dist"], WRSN_S_NBR_ESEND=st["nbr_esend"], WRSN_S_NBR_PTR=ptr_n,
                        WRSN_S_TGT_PTR=ptr_t, WRSN_S_NBR_IDX=st["nbr_idx"], WRSN_S_TGT_IDX=st["tgt_idx"],
                        WRSN_S_DIRECT=st["direct"])
            for name, dt, size in _S_FIELDS:
                off = int(self._soff[E[name]])
                a = np.zeros(sizes[size], _NP[dt])
                v = np.asarray(vals[name], _NP[dt])
                a[:len(v)] = v
                buf[s, off:off + a.nbytes] = a.view(np.uint8)
        return buf

    def _view(self, state, field, dtype, count):
        off = int(self._foff[self.E[field]])
        nbytes = count * torch.empty((), dtype=dtype).element_size()
        return state[:, off:off + nbytes].view(dtype)

    def _mask_ptr(self, mask):
        if mask is None:
            return None, None
        m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        return m, C.c_void_p(m.data_ptr())

    def _make_snapshot(self):
        """The state at t = warm_up is a pure function of the scenario (SURVEY Q8): simulate the warm-up once per
        scenario on the device and let ``reset`` restore it (``wrsn_reset_from_snapshot``)."""
        d = self.dims
        ds = _lib.Dims.from_buffer_copy(d)
        ds.B = d.n_scen
        snap = torch.zeros((d.n_scen, d.state_bytes), dtype=torch.uint8, device=self.device)
        ids = torch.arange(d.n_scen, dtype=torch.int32, device=self.device)
        until = torch.full((d.n_scen,), self.warm_up_time, dtype=torch.float64, device=self.device)
        L, st = self.L, self._stream()
        self._call(L.wrsn_init_network, C.byref(ds), self.scen.data_ptr(), ids.data_ptr(), snap.data_ptr(), None, 1, st)
        self._call(L.wrsn_run_until, C.byref(ds), self.scen.data_ptr(), ids.data_ptr(), snap.data_ptr(), None,
                                    until.data_ptr(), st)
        self._sync()
        self._snap = snap

    # ------------------------------------------------------------------ the WRSN interface, batched
    def reset(self, mask=None):
        """``WRSN.reset`` (:41-83) for the selected environments (all when ``mask`` is None)."""
        m, mp = self._mask_ptr(mask)
        L = self.L
        self._call(L.wrsn_reset_from_snapshot, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                              self.state.data_ptr(), self._snap.data_ptr(), mp, C.byref(self.req.c),
                                              self._stream())
        return self.req

    def step(self, agent_id, action, mask=None):
        """``WRSN.step`` (:289-330).  ``agent_id``: int32[B] (-1 = None), ``action``: float64[B, 3]."""
        L = self.L
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        x = torch.as_tensor(action, device=self.device).to(torch.float64).contiguous()
        if a.shape != (self.B,) or x.shape != (self.B, 3):
            raise ValueError("agent_id must be [B], action [B, 3]")
        m, mp = self._mask_ptr(mask)
        self._call(L.wrsn_step, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(), self.state.data_ptr(),
                               mp, a.data_ptr(), x.data_ptr(), C.byref(self.req.c), self._stream())
        return self.req

    def rollout_step(self, action, obs=None):
        """The rollout loop body of the reference's trainers (``controller/ippo/IPPO.py:137-143``) for every environment
        in one call and three kernel launches: ``step`` where the last request named a deciding charger (with
        ``action[b]``), ``reset`` where the episode has just ended, then ``get_state`` of every deciding charger into
        ``obs`` ([B, 4, S, S] float32 / float64; skipped when None).  No host synchronisation, no temporaries."""
        if action.dtype != torch.float64 or not action.is_contiguous() or action.shape != (self.B, 3) or action.device != self.state.device:
            raise ValueError("action must be a contiguous float64 tensor [B, 3] on the simulator's device")
        op, f64 = None, 0
        if obs is not None:
            if obs.dtype not in (torch.float32, torch.float64) or not obs.is_contiguous() or obs.shape != (self.B, 4, self.S, self.S):
                raise ValueError("obs must be a contiguous float32/float64 tensor [B, 4, S, S]")
            op, f64 = obs.data_ptr(), 1 if obs.dtype == torch.float64 else 0
        self._call(self.L.wrsn_rollout_step, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                            self.state.data_ptr(), self._snap.data_ptr(), action.data_ptr(),
                                            C.byref(self.req.c), op, f64, self._stream())
        return self.req

    def get_state(self, agent_id=None, out=None, dtype=torch.float32):
        """``WRSN.get_state`` (:130-186) of charger ``agent_id[b]`` in every environment with ``agent_id[b] >= 0``
        (default: the deciding charger of the last request), written to ``out`` [B, 4, S, S]."""
        if agent_id is None:
            agent_id = self.req.agent_id
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        if out is None:
            out = torch.zeros((self.B, 4, self.S, self.S), dtype=dtype, device=self.device)
        if out.dtype not in (torch.float32, torch.float64) or not out.is_contiguous() or out.shape != (self.B, 4, self.S, self.S):
            raise ValueError("out must be a contiguous float32/float64 tensor [B, 4, S, S]")
        self._call(self.L.wrsn_observe, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                       self.state.data_ptr(), a.data_ptr(), out.data_ptr(),
                                       1 if out.dtype == torch.float64 else 0, self._stream())
        return out

    def density_map_to_action(self, dmap, agent_id=None, out=None):
        """``WRSN.density_map_to_action`` (:229-287) with the map normalisation of ``WRSN.step`` (:293-296) for every
        environment with ``agent_id[b] >= 0`` (default: the deciding charger of the last request): ``dmap`` [B, S, S]
        float32 / float64 in HBM -> actions [B, 3] float64 (x-frac, y-frac, charge-time frac), ready for ``step`` /
        ``rollout_step``.  One streaming pass over the maps, no host round trip."""
        if agent_id is None:
            agent_id = self.req.agent_id
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        if dmap.dtype not in (torch.float32, torch.float64) or not dmap.is_contiguous() or dmap.shape != (self.B, self.S, self.S) \
                or dmap.device != self.state.device:
            raise ValueError("dmap must be a contiguous float32/float64 tensor [B, S, S] on the simulator's device")
        if out is None:
            out = torch.zeros((self.B, 3), dtype=torch.float64, device=self.device)
        if out.dtype != torch.float64 or not out.is_contiguous() or out.shape != (self.B, 3):
            raise ValueError("out must be a contiguous float64 tensor [B, 3]")
        self._call(self.L.wrsn_decode_density_map, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                                  self.state.data_ptr(), a.data_ptr(), dmap.data_ptr(),
                                                  1 if dmap.dtype == torch.float64 else 0, out.data_ptr(), self._stream())
        return out

    def linear_controller_action(self, obs, weights, agent_id=None, out=None):
        """``density_map_to_action`` for a controller whose map is a linear combination of the observation's channels — the
        reference's RandomController is ``weights = (1, 1, -10, 1)`` (``controller/random/RandomController.py:12-15``) —
        without materialising the map: ``obs`` [B, C, S, S] float32 in HBM -> actions [B, 3] float64.  Equal, bit for bit, to
        ``density_map_to_action(w0 * obs[:, 0] + w1 * obs[:, 1] + ...)`` evaluated by torch in float32."""
        if agent_id is None:
            agent_id = self.req.agent_id
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        if obs.dtype != torch.float32 or not obs.is_contiguous() or obs.dim() != 4 or obs.shape[0] != self.B \
                or obs.shape[2:] != (self.S, self.S) or obs.device != self.state.device:
            raise ValueError("obs must be a contiguous float32 tensor [B, C, S, S] on the simulator's device")
        w = (C.c_float * obs.shape[1])(*[float(x) for x in weights])
        if len(w) != obs.shape[1]:
            raise ValueError("one weight per channel")
        if out is None:
            out = torch.zeros((self.B, 3), dtype=torch.float64, device=self.device)
        if out.dtype != torch.float64 or not out.is_contiguous() or out.shape != (self.B, 3):
            raise ValueError("out must be a contiguous float64 tensor [B, 3]")
        self._call(self.L.wrsn_decode_linear_controller, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                   self.state.data_ptr(), a.data_ptr(), obs.data_ptr(), int(obs.shape[1]), w, out.data_ptr(), self._stream())
        return out

    def heuristic_action(self, kind="min_lifetime", agent_id=None, out=None):
        """A hand-written charging decision (``wrsn_heuristic_action``) for every environment with ``agent_id[b] >= 0`` (default:
        the deciding charger of the last request), computed from the state record: ``kind`` is one of ``HEURISTICS``,
        ``"min_lifetime"`` (the alive node with the lowest lifetime ``(energy - threshold) / energyCS`` that no other living
        charger is headed for) or ``"nearest_urgent"`` (the nearest such node among those that die within one worst-case move
        plus full charge; otherwise as ``"min_lifetime"``).  -> actions [B, 3] float64 (x-frac, y-frac, charge-time frac) on
        the device, ready for ``step`` / ``rollout_step``; the other rows of ``out`` are left untouched."""
        if kind not in HEURISTICS:
            raise ValueError("kind must be one of %s, not %r" % (", ".join(HEURISTICS), kind))
        if agent_id is None:
            agent_id = self.req.agent_id
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        if a.shape != (self.B,):
            raise ValueError("agent_id must be [B]")
        if out is None:
            out = torch.zeros((self.B, 3), dtype=torch.float64, device=self.device)
        if out.dtype != torch.float64 or not out.is_contiguous() or out.shape != (self.B, 3) or out.device != self.state.device:
            raise ValueError("out must be a contiguous float64 tensor [B, 3] on the simulator's device")
        self._call(self.L.wrsn_heuristic_action, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                   self.state.data_ptr(), a.data_ptr(), HEURISTICS.index(kind), out.data_ptr(), self._stream())
        return out

    def heuristic_candidates(self, kind="min_lifetime", width=8, agent_id=None, out=None, node=None):
        """The rule's ``width`` best candidates (``wrsn_heuristic_candidates``) for every environment with a deciding charger
        ``agent_id[b] >= 0`` (default: that of the last request): the first ``width`` nodes of ``heuristic_action``'s candidate
        set in the rule's order (``"min_lifetime"``: lowest lifetime first; ``"nearest_urgent"``: the urgent nodes nearest
        first, then the rest by lifetime).  -> (actions [B, width, 3] float64, nodes [B, width] int32), slot 0 being
        ``heuristic_action``'s decision bit for bit.  Slots beyond the row's candidate count hold node -1 and slot 0's action;
        the other rows of ``out`` / ``node`` are left untouched.  ``width``: 1 to ``WRSN_CAND_MAX`` (32)."""
        if kind not in HEURISTICS:
            raise ValueError("kind must be one of %s, not %r" % (", ".join(HEURISTICS), kind))
        K = int(width)
        if not 1 <= K <= self.E["WRSN_CAND_MAX"]:
            raise ValueError("width must lie in [1, %d], not %d" % (self.E["WRSN_CAND_MAX"], K))
        if agent_id is None:
            agent_id = self.req.agent_id
        a = torch.as_tensor(agent_id, device=self.device).to(torch.int32).contiguous()
        if a.shape != (self.B,):
            raise ValueError("agent_id must be [B]")
        if out is None:
            out = torch.zeros((self.B, K, 3), dtype=torch.float64, device=self.device)
        if node is None:
            node = torch.full((self.B, K), -1, dtype=torch.int32, device=self.device)
        if out.dtype != torch.float64 or not out.is_contiguous() or out.shape != (self.B, K, 3) or out.device != self.state.device:
            raise ValueError("out must be a contiguous float64 tensor [B, width, 3] on the simulator's device")
        if node.dtype != torch.int32 or not node.is_contiguous() or node.shape != (self.B, K) or node.device != self.state.device:
            raise ValueError("node must be a contiguous int32 tensor [B, width] on the simulator's device")
        self._call(self.L.wrsn_heuristic_candidates, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                   self.state.data_ptr(), a.data_ptr(), HEURISTICS.index(kind), K, out.data_ptr(), node.data_ptr(), self._stream())
        return out, node

    def rule_rollout(self, kind, limit, first_action=None, running=None, decisions=None, returns=None, launch_max=None):
        """Continue the rows ``running`` (bool [B]; default: every row whose request names a deciding charger) under the rule
        ``kind`` (one of ``HEURISTICS``) until each one's episode ends (``agent_id == -1``) or, at a request that is not in flight,
        it has made ``limit`` decisions — ``controllers.evaluate``'s accounting (``episode_ends``, ``episode_step``), run on the
        device by ``wrsn_rule_rollout``: the rule decides inside the step kernel and the row keeps stepping.  A row's first
        decision (``decisions[b] == 0``) takes ``first_action[b]`` ([B, 3] float64) when given.  ``decisions`` (int64 [B]) counts
        the actions handed out and ``returns`` (float64 [B]) adds the reward of every request after a step (NaN counted as 0);
        both start at 0 unless given, and are updated in place when given.  Each launch hands out at most ``launch_max`` (default
        1024) decisions per row; the dims' ``step_budget`` bounds the work of a whole launch.  One host synchronisation per
        launch, then ``raise_on_error``.  -> (returns, decisions, running), ``running`` all False; the request record holds
        every row's last request."""
        if kind not in HEURISTICS:
            raise ValueError("kind must be one of %s, not %r" % (", ".join(HEURISTICS), kind))
        limit = int(limit)
        lm = 1024 if launch_max is None else int(launch_max)
        if limit < 0:
            raise ValueError("limit must not be negative")
        if not 1 <= lm <= self.E["WRSN_ROLL_MAX"]:
            raise ValueError("launch_max must lie in [1, %d], not %d" % (self.E["WRSN_ROLL_MAX"], lm))
        B, dev = self.B, self.state.device

        def own(x, dtype, shape, name, default):
            if x is None:
                return default()
            if x.dtype != dtype or not x.is_contiguous() or tuple(x.shape) != shape or x.device != dev:
                raise ValueError("%s must be a contiguous %s tensor %s on the simulator's device" % (name, str(dtype)[6:], list(shape)))
            return x

        fa = None
        if first_action is not None:
            fa = own(first_action, torch.float64, (B, 3), "first_action", None)
        dec = own(decisions, torch.int64, (B,), "decisions", lambda: torch.zeros(B, dtype=torch.int64, device=dev))
        ret = own(returns, torch.float64, (B,), "returns", lambda: torch.zeros(B, dtype=torch.float64, device=dev))
        if running is None:
            run = (self.req.agent_id >= 0).to(torch.uint8)
        else:
            if running.shape != (B,) or running.device != dev or running.dtype not in (torch.bool, torch.uint8):
                raise ValueError("running must be a bool / uint8 tensor [B] on the simulator's device")
            run = running.to(torch.uint8).contiguous()
        while bool(run.any()):                           # one host synchronisation per launch
            self._call(self.L.wrsn_rule_rollout, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                       self.state.data_ptr(), run.data_ptr(), HEURISTICS.index(kind), None if fa is None else fa.data_ptr(),
                       limit, lm, dec.data_ptr(), ret.data_ptr(), C.byref(self.req.c), self._stream())
        self.raise_on_error()
        return ret, dec, run.to(torch.bool)

    def _branch(self, K):
        """The branch batch of ``lookahead`` for ``K`` candidates: B * K rows of this batch's scenarios and settings."""
        br = self._branches.get(K)
        if br is None:
            d = self.dims
            br = BatchedWRSN(self.scenarios, num_agent=self.num_agent, mc_type=self.mc_type, num_envs=self.B * K, map_size=self.map_size,
                             warm_up_time=self.warm_up_time, device=self.device, threads=d.threads, step_budget=d.step_budget,
                             step_rounds=d.step_rounds)
            self._branches[K] = br
        return br

    def lookahead(self, candidates, horizon, rollout_kind="min_lifetime", valid=None):
        """The value of each candidate action of each environment's deciding charger: for every row b whose request names a
        charger and every slot k with ``valid[b, k]`` (default all), a copy of the row (``wrsn_copy_rows``) is stepped once with
        ``candidates[b, k]`` ([B, K, 3] float64, any actions), then under the rule ``rollout_kind`` until it has made
        ``horizon`` more decisions or its episode has ended, with ``controllers.evaluate``'s accounting (``episode_ends``,
        ``episode_step``).  -> values [B, K] float64: the sum of the rewards of the branch's requests; -inf for a slot that is
        not valid, NaN for every slot of a row without a deciding charger.  Those cost no branch work.

        The branches are the rows of a second batch of B * K rows with this batch's scenarios and settings, built at the first
        call with K candidates and reused, and run by one ``rule_rollout`` of ``horizon + 1`` decisions that starts with the
        candidates.  This batch is not changed.  Host synchronisations: one per launch of the rollout (one when no branch runs
        into the step budget or past 1024 decisions), and ``raise_on_error`` of the branch batch at the end."""
        c = candidates
        if c.dtype != torch.float64 or not c.is_contiguous() or c.dim() != 3 or c.shape[0] != self.B or c.shape[2] != 3 \
                or not 1 <= c.shape[1] or c.device != self.state.device:
            raise ValueError("candidates must be a contiguous float64 tensor [B, K, 3] on the simulator's device")
        if rollout_kind not in HEURISTICS:
            raise ValueError("rollout_kind must be one of %s, not %r" % (", ".join(HEURISTICS), rollout_kind))
        H = int(horizon)
        if H < 0:
            raise ValueError("horizon must not be negative")
        B, K = self.B, int(c.shape[1])
        if valid is None:
            valid = torch.ones((B, K), dtype=torch.bool, device=self.device)
        valid = torch.as_tensor(valid, device=self.device).to(torch.bool)
        if valid.shape != (B, K):
            raise ValueError("valid must be [B, K]")
        br = self._branch(K)
        aid = self.req.agent_id
        decider = (aid >= 0) & (aid < self.M)
        running = (decider[:, None] & valid).reshape(B * K)
        rows = torch.arange(B * K, dtype=torch.int32, device=self.device)
        src = torch.where(running, rows // K, torch.full_like(rows, -1))     # -1: skipped by the copy
        self._call(self.L.wrsn_copy_rows, C.byref(self.dims), B * K, self.state.data_ptr(), C.byref(self.req.c), self.scen_id.data_ptr(),
                   src.data_ptr(), B, br.state.data_ptr(), C.byref(br.req.c), br.scen_id.data_ptr(), rows.data_ptr(), B * K,
                   self._stream())
        br._refresh_counts()
        ret, _, _ = br.rule_rollout(rollout_kind, H + 1, first_action=c.reshape(B * K, 3), running=running)
        val = torch.where(valid, ret.view(B, K), torch.full_like(ret.view(B, K), -math.inf))
        return torch.where(decider[:, None], val, torch.full_like(val, math.nan))

    def get_network_fitness(self):
        """``WRSN.get_network_fitness`` (:188-220): per-target values [B, T] and their minimum [B] over each row's own
        targets (columns beyond a row's own target count stay 0)."""
        fit = torch.zeros((self.B, max(self.T, 1)), dtype=torch.float64, device=self.device)
        mn = torch.zeros((self.B,), dtype=torch.float64, device=self.device)
        self._call(self.L.wrsn_fitness, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                       self.state.data_ptr(), fit.data_ptr(), mn.data_ptr(), self._stream())
        return fit[:, :self.T], mn

    # ------------------------------------------------------------------ copies of running environments (wrsn_copy_rows)
    def _rows(self, rows, what):
        """Host copy of a row list, every index in [0, B)."""
        r = np.asarray(rows.cpu() if isinstance(rows, torch.Tensor) else rows, np.int64).reshape(-1)
        if r.size and (r.min() < 0 or r.max() >= self.B):
            raise ValueError("%s: row indices must lie in [0, %d)" % (what, self.B))
        return r

    def _copy_rows(self, src, src_rows, dst, dst_rows):
        """``wrsn_copy_rows`` from ``src`` to ``dst``, each (state, wrsn_request, scen_id); the host row lists are the caller's,
        already checked."""
        n = len(src_rows)
        if n == 0:
            return
        sr = torch.as_tensor(src_rows.astype(np.int32), device=self.device)
        dr = torch.as_tensor(dst_rows.astype(np.int32), device=self.device)
        (ss, sq, si), (ds, dq, di) = src, dst
        self._call(self.L.wrsn_copy_rows, C.byref(self.dims), n, ss.data_ptr(), C.byref(sq), si.data_ptr(), sr.data_ptr(),
                   int(ss.shape[0]), ds.data_ptr(), C.byref(dq), di.data_ptr(), dr.data_ptr(), int(ds.shape[0]), self._stream())

    def _refresh_counts(self):
        if self._counts is None:                         # node and target count of every scenario
            self._counts = torch.as_tensor([[st["N"] for st in self.statics], [st["T"] for st in self.statics]], dtype=torch.int32,
                                           device=self.device)
        sid = self.scen_id.long()
        self.num_nodes.copy_(self._counts[0][sid])
        self.num_targets.copy_(self._counts[1][sid])

    @property
    def fingerprints(self):
        """One ``snapshot.scenario_fingerprint`` per scenario of the batch."""
        if self._fingerprints is None:
            self._fingerprints = [scenario_fingerprint(st) for st in self.statics]
        return self._fingerprints

    def fork(self, src, dst):
        """Copy the running environments ``src[i]`` onto rows ``dst[i]`` (state record, scenario and request row: see
        ``wrsn_copy_rows``); each copy then continues exactly as its source would with the same actions, including a step in
        flight (``agent_id == -4``).  ``dst`` rows must be distinct and disjoint from ``src``.  A destination row of another
        scenario takes the source's (``num_nodes`` / ``num_targets`` follow)."""
        s, d = self._rows(src, "src"), self._rows(dst, "dst")
        if len(s) != len(d):
            raise ValueError("src and dst must have the same length (%d != %d)" % (len(s), len(d)))
        if len(np.unique(d)) != len(d):
            raise ValueError("dst: rows must be distinct")
        if np.intersect1d(s, d).size:
            raise ValueError("dst: rows %s are also in src" % np.intersect1d(s, d)[:8].tolist())
        me = (self.state, self.req.c, self.scen_id)
        self._copy_rows(me, s, me, d)
        self._refresh_counts()

    def snapshot(self, rows=None, base=0):
        """The continuation state of ``rows`` (default all) as an ``EnvSnapshot`` on this batch's device.  ``base`` is the
        global index of local row 0 (a shard passes the start of its ``sharding.shard_range``): the snapshot records global
        row ids."""
        r = np.arange(self.B, dtype=np.int64) if rows is None else self._rows(rows, "rows")
        n = len(r)
        q = Requests(n, self.device)
        req = {f: getattr(q, f) for f in REQ_FIELDS}
        state = torch.zeros((n, self.dims.state_bytes), dtype=torch.uint8, device=self.device)
        scen = torch.zeros((n,), dtype=torch.int32, device=self.device)
        self._copy_rows((self.state, self.req.c, self.scen_id), r, (state, c_request(req), scen), np.arange(n, dtype=np.int64))
        meta = layout_meta(self.L, self.dims, self._foff, self.fingerprints)
        return EnvSnapshot(meta, torch.as_tensor(r + int(base), dtype=torch.int64, device=self.device), scen, state, req)

    def restore(self, snap, rows=None, base=0):
        """Write the rows of ``snap`` into this batch.  ``rows=None``: every snapshot row whose global id lies in
        [base, base + B) goes to local row id - base; otherwise ``rows[i]`` receives the snapshot's row i.  Scenarios are
        matched by fingerprint (the batch may list them in another order).  Raises ValueError, naming the field, for a
        snapshot this batch cannot continue exactly: another ABI version, layout dim or offset, a scenario the batch does not
        have, bad lengths or indices.  Returns the request record."""
        snap.validate()
        check_layout(snap.meta, self.L.wrsn_abi_version(), {k: getattr(self.dims, k) for k in LAYOUT_DIMS}, list(self._foff))
        if rows is None:
            ids = snap.ids.cpu().numpy()
            sel = (ids >= int(base)) & (ids < int(base) + self.B)
            src, dst = np.nonzero(sel)[0], ids[sel] - int(base)
        else:
            dst = self._rows(rows, "rows")
            if len(dst) != len(snap):
                raise ValueError("rows: %d rows for a snapshot of %d" % (len(dst), len(snap)))
            src = np.arange(len(snap), dtype=np.int64)
        if len(np.unique(dst)) != len(dst):
            raise ValueError("rows: a destination row is written twice (duplicate global ids or rows)")
        mine = {fp: k for k, fp in enumerate(self.fingerprints)}
        table = np.array([mine.get(fp, -1) for fp in snap.meta["fingerprints"]], np.int32)
        used = np.unique(snap.scen.cpu().numpy()[src])
        absent = [int(k) for k in used if table[k] < 0]
        if absent:
            raise ValueError("fingerprints: scenario %d of the snapshot (%s) is not in this batch"
                             % (absent[0], snap.meta["fingerprints"][absent[0]][:16]))
        if snap.device != self.device:
            snap = snap.to(self.device)
        scen = torch.as_tensor(table, device=self.device)[snap.scen.long()].contiguous()
        self._copy_rows((snap.state, c_request(snap.req), scen), src, (self.state, self.req.c, self.scen_id), dst)
        self._refresh_counts()
        return self.req

    # ------------------------------------------------------------------ lower-level entry points (tests / profiling)
    def init_network(self, with_reward_process=True, mask=None):
        m, mp = self._mask_ptr(mask)
        self._call(self.L.wrsn_init_network, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                            self.state.data_ptr(), mp, 1 if with_reward_process else 0, self._stream())

    def run_until(self, t, mask=None):
        m, mp = self._mask_ptr(mask)
        tt = torch.as_tensor(t, dtype=torch.float64, device=self.device)
        if tt.ndim == 0:
            tt = tt.expand(self.B)
        tt = tt.contiguous()
        self._call(self.L.wrsn_run_until, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                         self.state.data_ptr(), mp, tt.data_ptr(), self._stream())

    def reset_finish(self, mask=None):
        m, mp = self._mask_ptr(mask)
        self._call(self.L.wrsn_reset_finish, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                            self.state.data_ptr(), mp, C.byref(self.req.c), self._stream())
        return self.req

    def charge_rates(self, charging=None, out=None):
        """The node x charger charging model, dense (``wrsn_k_charge``; ``Node.charger_connection`` ``Node.py:134-139`` over
        the ``connected_nodes`` of ``MobileCharger.charge`` ``MobileCharger.py:56-59``): the ``energyRR`` every alive node
        would receive [B, N] and the ``chargingRate`` every charger would draw [B, M] if the chargers selected by
        ``charging`` (uint8 [B, M]; default all) charged at their present positions.  Does not touch the state.  The columns
        of [B, N] beyond a row's own node count are not written."""
        if out is not None:                              # (node [B, N], mc [B, max(M, 1)]) of an earlier call, reused
            node, mc = out[0], out[1] if out[1].shape[1] == max(self.M, 1) else None
        else:
            node = torch.zeros((self.B, self.N), dtype=torch.float64, device=self.device)
            mc = torch.zeros((self.B, max(self.M, 1)), dtype=torch.float64, device=self.device)
        ch, cp = None, None
        if charging is not None:
            ch = torch.as_tensor(charging, device=self.device).to(torch.uint8).contiguous()
            if ch.shape != (self.B, self.M):
                raise ValueError("charging must be [B, M]")
            cp = C.c_void_p(ch.data_ptr())
        self._call(self.L.wrsn_k_charge, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(), self.state.data_ptr(),
                                        cp, node.data_ptr(), mc.data_ptr(), self._stream())
        return node, mc[:, :self.M]

    def kernel(self, name):
        """Standalone per-tick kernels: 'bfs', 'drain', 'bookkeep', 'reward'."""
        self._call(getattr(self.L, "wrsn_k_" + name), C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                   self.state.data_ptr(), self._stream())

    # ------------------------------------------------------------------ typed views of the state records (no copies)
    def view(self, name, state=None):
        st = self.state if state is None else state
        d, E = self.dims, self.E
        f64, i16, u8, i32 = torch.float64, torch.int16, torch.uint8, torch.int32
        if name in ("energy", "rr", "cs", "esend", "logc", "logtick"):
            return self._view(st, "WRSN_F_" + name.upper(), f64, d.Npad)[:, :self.N]
        if name in ("nbef", "naft", "level", "parent"):
            return self._view(st, "WRSN_F_" + name.upper(), i16, d.Npad)[:, :self.N]
        if name == "status":
            return self._view(st, "WRSN_F_STATUS", u8, d.Npad)[:, :self.N]
        if name == "hdr":
            return self._view(st, "WRSN_F_HDR", f64, E["WRSN_H_LEN"])
        if name == "mc":
            return self._view(st, "WRSN_F_MC", f64, max(self.M, 1) * E["WRSN_MC_LEN"]).view(st.shape[0], max(self.M, 1), E["WRSN_MC_LEN"])
        if name == "proc":
            return self._view(st, "WRSN_F_PROC", f64, d.n_slot * E["WRSN_PR_LEN"]).view(st.shape[0], d.n_slot, E["WRSN_PR_LEN"])
        if name == "ring":
            return self._view(st, "WRSN_F_RING", f64, E["WRSN_RING"] * d.Npad).view(st.shape[0], E["WRSN_RING"], d.Npad)[:, :, :self.N]
        if name == "tact_words":
            return self._view(st, "WRSN_F_TACT", i32, d.Tw)
        if name == "conn_words":
            return self._view(st, "WRSN_F_CONN", i32, max(self.M, 1) * d.W).view(st.shape[0], max(self.M, 1), d.W)
        raise KeyError(name)

    def hdr(self, field):
        return self.view("hdr")[:, self.E["WRSN_H_" + field]]

    def mc(self, field):
        return self.view("mc")[:, :self.M, self.E["WRSN_MC_" + field]]

    @property
    def now(self):
        return self.hdr("NOW")

    @property
    def alive(self):
        return self.hdr("ALIVE").to(torch.uint8)

    def targets_active(self):
        """``Network.targets_active`` as uint8 [B, T]."""
        w = self.view("tact_words").to(torch.int64) & 0xFFFFFFFF
        bits = (w.unsqueeze(-1) >> torch.arange(32, device=self.device)) & 1
        return bits.reshape(w.shape[0], -1)[:, :self.T].to(torch.uint8)

    def raise_on_error(self):
        """One host synchronisation: raise if any environment has EVER reported an engine error (``flags`` bit 1: e.g. the
        process slots overflowed) — also one that ``rollout_step`` has reset since; returns the number of environments that have
        seen every charger dead (bit 0; the reference never returns from such a step, here the episode is reset).  The batched
        rollouts call it once per window (``controllers.rollout``, ``IPPORollout.collect`` through ``BatchedIPPO.roll_out``)."""
        s = self.req.sticky
        both = torch.stack([(s & 2).ne(0).sum(), (s & 1).ne(0).sum()]).tolist()
        if both[0]:
            bad = torch.nonzero(s & 2).flatten()[:8].tolist()
            raise RuntimeError("wrsn_b200: engine error (flags bit 1) in %d environment(s), e.g. rows %s" % (both[0], bad))
        return int(both[1])

    def counters(self):
        """Device counters summed over environments: simulated seconds, events, serial (death) ticks, BFS runs, decisions."""
        h = self.view("hdr")
        E = self.E
        return {k: float(h[:, E["WRSN_H_" + n]].sum().item()) for k, n in
                (("ticks", "NTICKS"), ("events", "NEVENTS"), ("serial_ticks", "NSLOW"), ("bfs", "NBFS"),
                 ("stale_rebuilds", "NSTALE"), ("lazy_spans", "NLAZY"), ("batched_ticks", "NBATCH"), ("split_death_ticks", "NSPLIT"),
                 ("decisions", "NDECISIONS"))}
