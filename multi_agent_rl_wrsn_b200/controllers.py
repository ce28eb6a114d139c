"""Caller side of the hot path, batched: the reference's RandomController and the rollout loop of its runners.

``controller/random/RandomController.py:12`` returns the density map ``s0 + s1 - 10 s2 + s3`` of the observation it is
handed; ``runner/checkRL.py:33-36`` loops ``make_action -> step`` until the episode ends.  Here both run for B
environments at once and nothing leaves HBM: the map is formed by torch from the observation tensor, decoded by
``wrsn_decode_density_map`` and consumed by ``wrsn_rollout_step`` (which also resets finished episodes, as the trainers'
loops do: ``controller/ippo/IPPO.py:137-143``).  Trainers (PPO / IPPO) plug in at the same place: anything with a
``make_action(agent_id, state)`` that returns either [B, S, S] maps or [B, 3] actions.
"""
import ctypes as C
import math

import torch

from . import _lib
from .batched import HEURISTICS, BatchedWRSN, episode_ends, episode_step
from .sharding import reduce_stats


class BatchedRandomController:
    """``RandomController.make_action`` for a batch: ``state`` is the [B, 4, S, S] observation tensor.  ``weights``: the map is
    this linear combination of the channels, which lets ``rollout`` decode it without materialising it
    (``BatchedWRSN.linear_controller_action``)."""
    weights = (1.0, 1.0, -10.0, 1.0)

    def make_action(self, agent_id, state, info=None, wrsn=None):
        return state[:, 0] + state[:, 1] - 10.0 * state[:, 2] + state[:, 3]


class HeuristicController:
    """A hand-written charging rule as a controller: ``kind`` is one of ``HEURISTICS`` (``BatchedWRSN.heuristic_action``).
    The decision is computed from the state record, not from the observation, so ``rollout`` and ``evaluate`` take it
    directly (``heuristic``) and render no observation for it."""

    def __init__(self, kind="min_lifetime"):
        if kind not in HEURISTICS:
            raise ValueError("kind must be one of %s, not %r" % (", ".join(HEURISTICS), kind))
        self.heuristic = kind

    def make_action(self, agent_id, state, info=None, wrsn=None):
        """Actions [B, 3] for the requests ``agent_id`` of ``wrsn`` (a ``BatchedWRSN``), or the 3-vector of charger ``agent_id``
        when ``wrsn`` is the single-environment ``WRSN``; ``state`` is not read."""
        if wrsn is None:
            raise ValueError("HeuristicController.make_action needs the environment (wrsn=)")
        if isinstance(wrsn, BatchedWRSN):
            return wrsn.heuristic_action(self.heuristic, agent_id=agent_id)
        return wrsn.heuristic_action(agent_id, self.heuristic)


class LookaheadController:
    """A rollout planner over a hand-written rule: at every decision it ranks the rule's ``width`` best nodes
    (``BatchedWRSN.heuristic_candidates``), tries each one at the rule's own charge fraction and then at each fraction of
    ``charge_levels`` (absolute, in [0, 1]), values every try by ``BatchedWRSN.lookahead`` (one step with it, then ``horizon``
    decisions of the rule ``kind``) and acts on the best.  Ties go to the lowest slot, so the rule's own decision (slot 0)
    wins them; with ``width=1`` and no ``charge_levels`` it decides as ``HeuristicController(kind)``.  ``rollout`` and
    ``evaluate`` take its action through ``plan``."""

    def __init__(self, kind="min_lifetime", width=8, horizon=4, charge_levels=()):
        if kind not in HEURISTICS:
            raise ValueError("kind must be one of %s, not %r" % (", ".join(HEURISTICS), kind))
        self.kind, self.width, self.horizon = kind, int(width), int(horizon)
        self.charge_levels = tuple(float(c) for c in charge_levels)
        if not all(0.0 <= c <= 1.0 for c in self.charge_levels):
            raise ValueError("charge_levels must lie in [0, 1]")
        self.last = None                                                  # (values, chosen slot) of the last plan

    def candidates(self, env):
        """-> (actions [B, K, 3], valid [B, K]) with K = width * (1 + len(charge_levels)): slot n * (1 + L) + l is the rule's
        n-th node at its own charge fraction (l = 0) or at ``charge_levels[l - 1]``.  Slot 0 is valid even without a node
        (the rule's stay action)."""
        act, node = env.heuristic_candidates(self.kind, self.width)
        L = len(self.charge_levels)
        act = act[:, :, None, :].expand(env.B, self.width, 1 + L, 3).clone()
        for l, c in enumerate(self.charge_levels):
            act[:, :, l + 1, 2] = c
        valid = (node >= 0)[:, :, None].expand(env.B, self.width, 1 + L).reshape(env.B, -1).clone()
        valid[:, 0] = True
        return act.reshape(env.B, -1, 3), valid

    def plan(self, env, out):
        """Write the planner's decision for every row of ``env`` (a ``BatchedWRSN``) with a deciding charger into ``out``
        [B, 3]; the other rows are left untouched."""
        cand, valid = self.candidates(env)
        values = env.lookahead(cand, self.horizon, self.kind, valid)
        best = torch.argmax(values, dim=1)                                # the first of equal maxima
        chosen = cand.gather(1, best[:, None, None].expand(env.B, 1, 3))[:, 0]
        out.copy_(torch.where((env.req.agent_id >= 0)[:, None], chosen, out))
        self.last = (values, best)
        return out


def rollout(env, controller, steps, obs=None, group=None):
    """``steps`` rollout steps of every environment of ``env`` (a ``BatchedWRSN``) under ``controller``.

    Returns the observation tensor and job-wide statistics (summed over ranks when torch.distributed is initialised:
    the only collective of the whole path): decisions handed out, simulated seconds, episodes finished, sum of rewards.
    A controller with ``plan`` (``LookaheadController``) or ``heuristic`` (``HeuristicController``) decides from the state
    record: its steps render no observation, and ``obs`` is filled once, after the last step.
    """
    B, S, dev = env.B, env.S, env.device
    plan = getattr(controller, "plan", None)
    heuristic = getattr(controller, "heuristic", None)
    from_state = plan is not None or heuristic is not None
    if obs is None:
        obs = torch.zeros((B, 4, S, S), dtype=torch.float32, device=dev)
        if not from_state:
            env.get_state(out=obs)
    action = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    local = torch.zeros(2, dtype=torch.float64, device=dev)               # episodes finished, sum of rewards
    resets0 = env.req.stats[:, 2].sum()
    dec0, sim0 = reduce_stats(env, group)
    fused = getattr(controller, "weights", None) is not None and obs.dtype == torch.float32
    for _ in range(int(steps)):
        if from_state:                                                    # action straight from the state record
            if plan is not None:
                plan(env, action)
            else:
                env.heuristic_action(heuristic, out=action)
            env.rollout_step(action)
            local[1] += torch.nan_to_num(env.req.reward, nan=0.0).sum()
            continue
        if fused:                                                         # map formed inside the decoder, channel by channel
            env.linear_controller_action(obs, controller.weights, out=action)
            env.rollout_step(action, obs)
            local[1] += torch.nan_to_num(env.req.reward, nan=0.0).sum()
            continue
        a = controller.make_action(env.req.agent_id, obs)
        if a.dim() == 3:                                                  # density maps: WRSN.step :293-297 on the device
            env.density_map_to_action(a.contiguous(), out=action)
        else:
            action.copy_(a)
        env.rollout_step(action, obs)
        local[1] += torch.nan_to_num(env.req.reward, nan=0.0).sum()
    if from_state:
        env.get_state(out=obs)
    local[0] = env.req.stats[:, 2].sum() - resets0                        # episodes that ended (and were reset) in these steps
    if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size(group) > 1:
        torch.distributed.all_reduce(local, group=group)
    dec1, sim1 = reduce_stats(env, group)
    all_dead = env.raise_on_error()                                       # engine errors of any step of the window, reset or not
    return obs, dict(decisions=dec1 - dec0, simulated_seconds=sim1 - sim0, episodes=float(local[0].item()),
                     reward_sum=float(local[1].item()), environments_that_saw_every_charger_dead=all_dead)


def evaluate(env, controller, episodes=1, max_decisions=None, check_every=16):
    """Run every environment of ``env`` (a ``BatchedWRSN``) from a reset under ``controller`` until it has finished
    ``episodes`` episodes, and report each one: the network lifetime and the return of a policy, as the papers compare them.

    An episode ends at a request that names no charger (``agent_id == -1``: the network is dead, ``terminal``, or every
    charger is), or — with ``max_decisions`` — at the first request after that many decisions (``truncated``).  Each row is
    stepped with ``step(mask=running)``, so its terminal request is read before ``reset(mask=finished)`` starts the next
    episode.  A request with no deciding charger that is not terminal (``agent_id == -2``) is stepped with agent -1; a step in
    flight (-4) continues.  The decision comes from ``plan(env, out)`` (``LookaheadController``) when the controller has one;
    a controller with ``heuristic`` (``HeuristicController``) runs each episode, for every row at once, as one
    ``BatchedWRSN.rule_rollout`` from the reset, which takes the same decisions without the per-request loop;
    otherwise from ``make_action(agent_id, obs)`` on the float32 observation (``get_state`` into one reused buffer), its maps
    decoded by ``density_map_to_action``, or by ``linear_controller_action`` when the controller has ``weights``.  A
    ``make_action`` that returns ``(action, log_prob)`` (a ``PerAgentPolicy``) is accepted.  The loop synchronises with the
    host once every ``check_every`` steps, to see whether any row is still running.

    Returns tensors [B, episodes] on the device: ``lifetime`` (``now`` at the episode's last request minus
    ``warm_up_time``), ``return`` (sum of the rewards of its requests, NaN counted as 0), ``decisions`` (actions handed to
    ``step``) and ``truncated``.
    """
    B, dev, E = env.B, env.device, int(episodes)
    if E < 1 or int(check_every) < 1:
        raise ValueError("episodes and check_every must be at least 1")
    cap = None if max_decisions is None else int(max_decisions)
    plan = getattr(controller, "plan", None)
    heuristic = getattr(controller, "heuristic", None)
    weights = getattr(controller, "weights", None)
    obs = None if heuristic is not None or plan is not None else torch.zeros((B, 4, env.S, env.S), dtype=torch.float32, device=dev)
    lifetime = torch.zeros((B, E), dtype=torch.float64, device=dev)
    ret = torch.zeros((B, E), dtype=torch.float64, device=dev)
    decisions = torch.zeros((B, E), dtype=torch.int64, device=dev)
    truncated = torch.zeros((B, E), dtype=torch.bool, device=dev)
    done = torch.zeros(B, dtype=torch.int64, device=dev)                 # episodes finished per row
    cur_ret = torch.zeros(B, dtype=torch.float64, device=dev)
    cur_dec = torch.zeros(B, dtype=torch.int64, device=dev)
    action = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    cols = torch.arange(E, device=dev)
    env.reset()
    if plan is None and heuristic is not None:
        for e in range(E):
            if e:
                env.reset()
            r, d, _ = env.rule_rollout(heuristic, 1 << 62 if cap is None else cap, running=torch.ones(B, dtype=torch.bool, device=dev))
            lifetime[:, e] = env.req.now - env.warm_up_time
            ret[:, e], decisions[:, e] = r, d
            truncated[:, e] = env.req.agent_id != -1
        return {"lifetime": lifetime, "return": ret, "decisions": decisions, "truncated": truncated}
    k = 0
    while True:
        req = env.req
        running = done < E
        fin_term, fin = episode_ends(req, running, cur_dec, cap)
        hit = fin[:, None] & (cols[None, :] == done[:, None])            # this episode's column
        lifetime.copy_(torch.where(hit, (req.now - env.warm_up_time)[:, None], lifetime))
        ret.copy_(torch.where(hit, cur_ret[:, None], ret))
        decisions.copy_(torch.where(hit, cur_dec[:, None], decisions))
        truncated.copy_(truncated | (hit & ~fin_term[:, None]))
        done += fin.to(torch.int64)
        cur_ret.masked_fill_(fin, 0.0)
        cur_dec.masked_fill_(fin, 0)
        running = done < E
        env.reset(mask=fin & running)
        if k % int(check_every) == 0 and not bool(running.any()):      # the loop's only host synchronisation
            break
        k += 1
        aid = req.agent_id
        if plan is not None:
            plan(env, action)
        else:
            env.get_state(out=obs)
            if weights is not None:
                env.linear_controller_action(obs, weights, out=action)
            else:
                a = controller.make_action(aid, obs)
                if isinstance(a, tuple):
                    a = a[0]
                if a.dim() == 3:
                    env.density_map_to_action(a.contiguous(), out=action)
                else:
                    action.copy_(a)
        episode_step(env, running, action, cur_dec, cur_ret)
    env.raise_on_error()
    return {"lifetime": lifetime, "return": ret, "decisions": decisions, "truncated": truncated}


class IPPORollout:
    """``IPPO.roll_out`` (``controller/ippo/IPPO.py:119-210``; ``PPO.roll_out`` is the same loop with one shared
    network) for B environments at once, with the record kept in HBM.

    The reference loops ``get_action -> step`` on one environment and, per agent, appends a transition
    ``(prev_state, input_action, log_prob, reward, state, terminal)`` whenever a request names an agent that has
    already acted in the current episode (``:141-155``); ``prev_state`` is the observation that agent was last handed.
    Here the T rollout steps are stored time-major (``obs[t]`` = the observation handed out at step t, one request per
    environment and step) and a transition is a *link*: ``link[t, b]`` is the earlier step at which environment b
    asked the same agent in the same episode, or -1.  Nothing is copied twice and nothing leaves the device:

        state = obs[link[t, b], b]   action, log_prob = act / logp[link[t, b], b]
        next_state = obs[t, b]       reward = reward[t, b]        terminal = False  (the reference breaks on terminal
                                                                                     before it records, ``:143-144``)

    ``policy(agent_id, obs)`` -> ``(input_action, log_prob)`` with ``agent_id`` int32 [B], ``obs`` [B, 4, S, S];
    ``input_action`` is a [B, S, S] density map (``density_map=True``, the runners' setting) or a [B, 3] action.
    """

    def __init__(self, env, steps, action_shape=None, obs_dtype=torch.float32, with_obs=True, keep_open=False):
        """``keep_open=True``: ``carry_over`` saves the decisions that are still open at the end of a window (observation, action,
        log-probability per environment and agent: B x M x 160 KB at map size 100), so that transitions whose request arrives in
        the next window are recorded too instead of being dropped at the window boundary.
        ``with_obs=False`` keeps no observations (``policy`` is handed None; ``batch`` has no states): for policies that
        do not look at the map, and for the CPU tests of the record, whose host emulation has no raster."""
        B, S, M, dev = env.B, env.S, env.M, env.device
        self.env, self.T = env, int(steps)
        action_shape = (S, S) if action_shape is None else tuple(action_shape)
        self.obs = torch.zeros((self.T + 1, B, 4, S, S), dtype=obs_dtype, device=dev) if with_obs else None
        self.now = torch.zeros((self.T + 1, B), dtype=torch.float64, device=dev)   # env.now of every request
        self.act = torch.zeros((self.T, B) + action_shape, dtype=torch.float32, device=dev)
        self.logp = torch.zeros((self.T, B), dtype=torch.float32, device=dev)
        self.reward = torch.zeros((self.T + 1, B), dtype=torch.float64, device=dev)
        self.agent = torch.full((self.T + 1, B), -1, dtype=torch.int64, device=dev)
        self.link = torch.full((self.T + 1, B), -1, dtype=torch.int64, device=dev)
        self.new_episode = torch.zeros((self.T + 1, B), dtype=torch.bool, device=dev)
        self.last = torch.full((B, M), -1, dtype=torch.int64, device=dev)   # step of each agent's open decision
        self.action = torch.zeros((B, 3), dtype=torch.float64, device=dev)
        self.terminal_factor = None
        self._collected = False
        self._resets = None
        self.keep_open = bool(keep_open)
        if self.keep_open:                                                # link == -2: the decision lives in these buffers
            self.open_obs = torch.zeros((B, M, 4, S, S), dtype=obs_dtype, device=dev) if with_obs else None
            self.open_act = torch.zeros((B, M) + action_shape, dtype=torch.float32, device=dev)
            self.open_logp = torch.zeros((B, M), dtype=torch.float32, device=dev)
            self.open_now = torch.zeros((B, M), dtype=torch.float64, device=dev)
        if bool((env.req.agent_id == -3).all()):                          # never reset: start the first episodes
            env.reset()
        if bool(((env.req.agent_id < 0) & (env.req.agent_id != -4)).any()):
            raise RuntimeError("IPPORollout needs an open request (a deciding charger) or a step in flight in every environment")
        if with_obs:
            env.get_state(out=self.obs[0])
        self.agent[0] = env.req.agent_id.to(torch.int64).clamp_min(-1)
        self.now[0] = env.req.now
        self._resets = env.req.stats[:, 2].clone()                       # episodes begun so far, per environment

    def collect(self, policy):
        """T rollout steps.  Row t of the record is the request answered at step t; row T is the request left open
        (its observation starts the next ``collect`` after ``carry_over``)."""
        env, L = self.env, self.env.L
        for t in range(self.T):
            a = self.agent[t]
            x, lp = policy(a.to(torch.int32), None if self.obs is None else self.obs[t])
            self.act[t].copy_(x)
            self.logp[t].copy_(lp)
            if x.dim() == 3:                                              # WRSN.step :293-297 on the device
                env.density_map_to_action(self.act[t], out=self.action)
            else:
                self.action.copy_(x)
            env.rollout_step(self.action, None if self.obs is None else self.obs[t + 1])
            # one launch for the loop's bookkeeping (:138-155): last[b, a] = t, cleared where the episode ended and was
            # reset; row t + 1 = the next request's agent, its link (-1: `continue`), reward and time
            _lib.check(L.wrsn_record_transitions(C.byref(env.dims), C.byref(env.req.c), t, a.data_ptr(), self.last.data_ptr(),
                                                 self._resets.data_ptr(), self.agent[t + 1].data_ptr(),
                                                 self.link[t + 1].data_ptr(), self.new_episode[t + 1].data_ptr(),
                                                 self.reward[t + 1].data_ptr(), self.now[t + 1].data_ptr(), env._stream()), L)
        self._collected = True
        return self

    def carry_over(self):
        """Start the next window from the open requests (the reference starts every ``roll_out`` with ``env.reset()``; a
        continuing batch keeps its episodes instead).  Decisions still open are saved and stay linkable with ``keep_open``,
        otherwise links into the finished window are dropped.  No-op on a fresh record."""
        if not self._collected:
            return
        self._collected = False
        if self.keep_open:                                                # save what the open decisions will be linked to
            fresh = self.last >= 0                                        # decided in the window that just ended
            at = self.last.clamp_min(0)                                   # [B, M] step of the decision
            rows = torch.arange(self.env.B, device=at.device)[:, None].expand_as(at)
            pick = lambda rec, buf: torch.where(fresh.reshape(fresh.shape + (1,) * (buf.dim() - 2)), rec[at, rows].to(buf.dtype), buf)
            if self.obs is not None:
                self.open_obs = pick(self.obs, self.open_obs)
            self.open_act, self.open_logp, self.open_now = pick(self.act, self.open_act), pick(self.logp, self.open_logp), pick(self.now, self.open_now)
            self.last = torch.where(fresh, torch.full_like(self.last, -2), self.last)   # -2 stays -2, -1 stays -1
        else:
            self.last.fill_(-1)
        if self.obs is not None:
            self.obs[0].copy_(self.obs[self.T])
        self.agent[0] = self.agent[self.T]
        self.now[0] = self.now[self.T]
        self.link.fill_(-1)
        self.new_episode.zero_()

    def transitions(self, agent_id):
        """Index tensors ``(t, b, t_prev)`` of the transitions recorded for ``agent_id``, in the reference's order
        inside every environment (time-major)."""
        sel = (self.agent[1:] == int(agent_id)) & (self.link[1:] != -1)        # -2: decided before this window (keep_open)
        t, b = torch.nonzero(sel, as_tuple=True)
        t = t + 1
        return t, b, self.link[t, b]

    def batch(self, agent_id, states=True, next_states=True):
        """The lists ``roll_out`` builds for one agent, as tensors (``:148-153``).  ``states`` / ``next_states`` = False leaves
        the (large) observation gathers out; ``tp`` / ``t`` / ``b`` index them in ``self.obs`` (``obs[tp, b]``, ``obs[t, b]``)."""
        t, b, tp = self.transitions(agent_id)
        a = int(agent_id)
        out = dict(actions=self._prev(self.act, "open_act", tp, b, a), log_probs=self._prev(self.logp, "open_logp", tp, b, a),
                   rewards=self.reward[t, b].to(torch.float32),
                   terminals=torch.zeros(t.shape, dtype=torch.float32, device=t.device), t=t, b=b, tp=tp,
                   prev_time=self._prev(self.now, "open_now", tp, b, a), time=self.now[t, b])
        if self.obs is not None and states:
            out["states"] = self._prev(self.obs, "open_obs", tp, b, a)
        if self.obs is not None and next_states:
            out["next_states"] = self.obs[t, b]
        return out

    def _prev(self, rec, open_name, tp, b, agent_id):
        """``rec[tp, b]``, or the saved open decision of ``agent_id`` where ``tp == -2`` (decided before this window)."""
        got = rec[tp.clamp_min(0), b]
        if not self.keep_open:
            return got
        saved = getattr(self, open_name)[b, agent_id].to(got.dtype)
        return torch.where((tp < -1).reshape((-1,) + (1,) * (got.dim() - 1)), saved, got)

    def cal_rt_adv(self, agent_id, value_fn, gamma, gae_lambda, gae=True, chunk=4096, values=None, next_values=None,
                   keep_states=True):
        """``IPPO.cal_rt_adv`` (``:71-94``) for every (environment, episode) sequence of ``agent_id`` at once.

        The reference evaluates the critic on an episode's states / next states and runs the recursion backwards over
        that episode's list with the recorded ``terminals`` as the continuation factor — which are all False
        (``:143-153``), so ``advantages = rewards - values`` and ``returns = rewards``; the recursion is kept general
        (``terminals`` may be overridden through ``self.terminal_factor``) and runs backwards over the T steps with
        one carry per environment, cleared where an episode begins.  ``values`` / ``next_values`` (one per transition of
        ``batch(agent_id)``) replace the critic calls when given.
        """
        bt = self.batch(agent_id, states=keep_states, next_states=False)
        n = bt["rewards"].shape[0]
        with torch.no_grad():
            if values is None:                       # the critic on states / next states, gathered chunk by chunk from the record
                cut = lambda x, i: x[i:i + chunk]
                ev = lambda get: torch.cat([value_fn(get(i)) for i in range(0, n, chunk)]) if n else bt["rewards"]
                values = ev(lambda i: self._prev(self.obs, "open_obs", cut(bt["tp"], i), cut(bt["b"], i), int(agent_id)))
                next_values = ev(lambda i: self.obs[cut(bt["t"], i), cut(bt["b"], i)])
            term = bt["terminals"] if self.terminal_factor is None else torch.full_like(bt["terminals"], self.terminal_factor)
            B, dev = self.env.B, values.device
            grid = lambda v: torch.zeros((self.T + 1, B), dtype=torch.float32, device=dev).index_put_((bt["t"], bt["b"]), v)
            has = torch.zeros((self.T + 1, B), dtype=torch.bool, device=dev).index_put_((bt["t"], bt["b"]), torch.ones(n, dtype=torch.bool, device=dev))
            r, v, nv, tm = grid(bt["rewards"]), grid(values), grid(next_values), grid(term)
            out = torch.zeros_like(r)
            carry = torch.zeros(B, dtype=torch.float32, device=dev)
            for t in range(self.T, 0, -1):
                if gae:                                                   # :77-82
                    cur = r[t] + gamma * nv[t] * tm[t] - v[t] + gamma * gae_lambda * tm[t] * carry
                else:                                                     # :84-91; the reference indexes returns[len] at the last
                                                                          # step of a list (IndexError): here the tail value is 0
                    cur = r[t] + gamma * tm[t] * carry
                out[t] = torch.where(has[t], cur, out[t])
                carry = torch.where(has[t], cur, carry)
                carry = torch.where(self.new_episode[t], torch.zeros_like(carry), carry)
            seq = out[bt["t"], bt["b"]]
            if gae:
                advantages, returns = seq, seq + values
            else:
                returns, advantages = seq, seq - values
        return returns, advantages, values, bt


def select_batch(rewards, batch_size, generator=None):
    """The reward-outlier batch selection of ``IPPO.roll_out`` (``:193-200``): the ``batch_size // 2`` transitions whose
    reward is farthest from the mean, plus ``batch_size - batch_size // 2`` drawn without replacement from the first
    ``len - batch_size // 2`` indices (of the *unsorted* list, as the reference does).  Index tensor on the rewards' device;
    the draw uses torch's generator, not numpy's global one."""
    n = rewards.shape[0]
    selected = int(batch_size / 2.0)
    random_num = int(batch_size) - selected
    if n - selected < random_num:
        raise ValueError("Cannot take a larger sample than population when 'replace=False'")   # np.random.choice's error
    order = torch.argsort((rewards - rewards.mean()).abs(), stable=True)
    gdev = rewards.device if generator is None else generator.device        # a generator draws on its own device
    draw = torch.randperm(n - selected, generator=generator, device=gdev)[:random_num].to(rewards.device)
    return torch.cat((order[n - selected:], draw))


class PerAgentPolicy:
    """``IPPO.get_action`` (``controller/ippo/IPPO.py:96-106``) for a batch of requests: IPPO keeps one actor per
    charger, so the requests are grouped by agent id and ``actors[i]`` runs once on its slice of the observation tensor
    (in HBM, no host copy); the action is a sample of ``Normal(mean, exp(log_std))`` and the log-probability its sum over
    the map, exactly what ``IPPO.evaluate`` (``:108-115``) recomputes during the update.  ``PPO`` (one shared network,
    ``controller/ppo/PPO.py``) is ``PerAgentPolicy([actor] * num_agent)``.  One host synchronisation per call: the sizes
    of the groups."""

    def __init__(self, actors, generator=None, action_shape=None, chunk=512):
        """``action_shape``: shape of one action — default the S x S density map of the reference's actors; ``(3,)`` for
        actors that emit the 3-vector action directly (``density_map=False``)."""
        self.actors, self.generator = list(actors), generator
        self.action_shape = None if action_shape is None else tuple(action_shape)
        self.chunk = int(chunk)                       # rows per forward pass (bounds the activations of a 4096-row batch)

    @torch.no_grad()
    def __call__(self, agent_id, obs):
        B, S = obs.shape[0], obs.shape[-1]
        M = len(self.actors)
        ids = agent_id.to(torch.int64).clamp_min(-1) + 1                 # 0: row without a request (step in flight), skipped
        order = torch.argsort(ids, stable=True)
        counts = torch.bincount(ids, minlength=M + 1).tolist()
        if len(counts) > M + 1:
            raise ValueError("request for agent %d but only %d actors" % (len(counts) - 2, M))
        skipped, counts = counts[0], counts[1:]
        shape = (S, S) if self.action_shape is None else self.action_shape
        red = tuple(range(1, 1 + len(shape)))
        x = torch.zeros((B,) + shape, dtype=torch.float32, device=obs.device)
        lp = torch.zeros((B,), dtype=torch.float32, device=obs.device)
        lo = skipped
        for i, n in enumerate(counts):
            if n == 0:
                continue
            for c0 in range(0, n, self.chunk):
                idx = order[lo + c0:lo + min(n, c0 + self.chunk)]
                m = int(idx.numel())
                mean, log_std = self.actors[i](obs[idx].to(torch.float32))
                mean, log_std = mean.reshape((m,) + shape), log_std.reshape((m,) + shape)   # UNet.forward squeezes a batch of one away
                std = log_std.exp()
                gdev = mean.device if self.generator is None else self.generator.device
                a = mean + std * torch.randn(mean.shape, generator=self.generator, device=gdev, dtype=mean.dtype).to(mean.device)
                logp = (-((a - mean) ** 2) / (2.0 * std * std) - log_std - 0.5 * math.log(2.0 * math.pi)).sum(red)   # Normal.log_prob
                x[idx] = a
                lp[idx] = logp
            lo += n
        return x, lp


def allreduce_gradients(parameters, group=None):
    """Average the gradients of ``parameters`` over the ranks of ``group`` with ONE all-reduce of a flat bucket (the
    reference's actor + critic pair is 8.3 MB: a single NCCL launch over NVLink / NVSwitch per minibatch; gloo in the CPU
    tests).  The only collective a trainer adds to the path — the simulation itself has none."""
    dist = torch.distributed
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    grads = [p.grad for p in parameters if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.div_(dist.get_world_size(group))
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


def ppo_update(actor, critic, optimizer, batch, args, group=None, generator=None, timers=None):
    """The update of one agent in ``IPPO.train`` (``controller/ippo/IPPO.py:222-268``; ``PPO.train`` is the same code):
    ``n_updates_per_iteration`` passes over ``batch`` (tensors of ``batch_size`` rows: states, actions, log_probs,
    advantages, returns, values) in shuffled minibatches, clipped surrogate + (clipped) value loss - entropy bonus,
    gradient-norm clipping of actor and critic separately, one optimizer step per minibatch.  ``args`` is the
    ``alg_args`` mapping of ``alg_args/ippo.yaml`` / ``ppo.yaml``.  With several ranks every rank passes its own shard's
    batch and the gradients are averaged before the clipping (``allreduce_gradients``), so all replicas stay identical.
    Returns the statistics the reference writes to TensorBoard (``:270-279``) for the last minibatch."""
    n = batch["states"].shape[0]
    mbs, clip = int(args["minibatch_size"]), float(args["clip"])
    params = list(actor.parameters()) + list(critic.parameters())
    clipfracs, stats = [], {}
    for _ in range(int(args["n_updates_per_iteration"])):
        gdev = "cpu" if generator is None else generator.device
        b_inds = torch.randperm(n, generator=generator, device=gdev).to(batch["states"].device)      # np.random.shuffle(b_inds), :229
        for start in range(0, n, mbs):
            mb = b_inds[start:start + mbs]
            m = mb.numel()
            states, actions = batch["states"][mb].to(torch.float32), batch["actions"][mb]
            mean, log_std = actor(states)                                               # IPPO.evaluate, :108-115
            mean, log_std = mean.reshape(actions.shape), log_std.reshape(actions.shape)
            dist_ = torch.distributions.Normal(mean, torch.exp(log_std))
            red = tuple(range(1, actions.dim()))
            newlogprob, entropy = dist_.log_prob(actions).sum(red), dist_.entropy().sum(red)
            newvalue = critic(states).sum(1).view(-1)                                   # IPPO.get_value, :117-119
            logratio = newlogprob - batch["log_probs"][mb]
            ratio = logratio.exp()
            with torch.no_grad():
                old_approx_kl = (-logratio).mean()
                approx_kl = ((ratio - 1) - logratio).mean()
                clipfracs.append(((ratio - 1.0).abs() > clip).float().mean())
            adv = batch["advantages"][mb]
            if args["norm_adv"]:
                adv = (adv - adv.mean()) / (adv.std() + 1e-8)
            pg_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
            ret, val = batch["returns"][mb], batch["values"][mb]
            if args["clip_vloss"]:
                v_clipped = val + torch.clamp(newvalue - val, -clip, clip)
                v_loss = 0.5 * torch.max((newvalue - ret) ** 2, (v_clipped - ret) ** 2).mean()
            else:
                v_loss = 0.5 * ((newvalue - ret) ** 2).mean()
            entropy_loss = entropy.mean()
            loss = pg_loss - float(args["ent_coef"]) * entropy_loss + v_loss * float(args["vf_coef"])
            optimizer.zero_grad()
            loss.backward()
            if timers is not None:                                                      # CUDA events around the collective
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
            allreduce_gradients(params, group)
            if timers is not None:
                ev[1].record()
                timers.append(ev)
            torch.nn.utils.clip_grad_norm_(actor.parameters(), float(args["max_grad_norm"]))
            torch.nn.utils.clip_grad_norm_(critic.parameters(), float(args["max_grad_norm"]))
            optimizer.step()
            stats = dict(loss=loss.detach(), value_loss=v_loss.detach(), policy_loss=pg_loss.detach(),
                         entropy=entropy_loss.detach(), old_approx_kl=old_approx_kl, approx_kl=approx_kl, minibatch=m)
    stats["clipfrac"] = torch.stack(clipfracs).mean() if clipfracs else None
    return stats
