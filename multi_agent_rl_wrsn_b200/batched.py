"""``BatchedWRSN`` — B independent WRSN environments advanced in lockstep on one B200.

Host-side mirror of ``rl_env.WRSN.WRSN`` (``rl_env/WRSN.py:21``): the same ``reset`` / ``step`` /
``get_state`` / ``get_network_fitness`` contract, but every argument and result carries a leading
environment axis and lives in HBM as a torch tensor.  All simulation work happens in the sm_100a kernels
behind the C ABI of ``include/wrsn_b200.h``; torch is the allocator and the stream provider only.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .scenario import Scenario, build_static, load_mc_type

_NP = {"f64": np.float64, "i32": np.int32, "u8": np.uint8}
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
        self.queue = torch.zeros((2,), dtype=torch.int32, device=device)       # work queue of the persistent step kernel (step_rounds < 0)
        self.c = _lib.Request(self.agent_id.data_ptr(), self.terminal.data_ptr(), self.reward.data_ptr(),
                              self.now.data_ptr(), self.action.data_ptr(), self.detail.data_ptr(), self.flags.data_ptr(),
                              self.stats.data_ptr(), self.sticky.data_ptr(), self.order.data_ptr(), self.queue.data_ptr())


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
        loop (same results, better instruction-cache behaviour; see include/wrsn_b200.h)."""
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

    def get_network_fitness(self):
        """``WRSN.get_network_fitness`` (:188-220): per-target values [B, T] and their minimum [B] over each row's own
        targets (columns beyond a row's own target count stay 0)."""
        fit = torch.zeros((self.B, max(self.T, 1)), dtype=torch.float64, device=self.device)
        mn = torch.zeros((self.B,), dtype=torch.float64, device=self.device)
        self._call(self.L.wrsn_fitness, C.byref(self.dims), self.scen.data_ptr(), self.scen_id.data_ptr(),
                                       self.state.data_ptr(), fit.data_ptr(), mn.data_ptr(), self._stream())
        return fit[:, :self.T], mn

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
