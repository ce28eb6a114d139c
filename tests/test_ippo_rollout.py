"""Batched IPPO rollout record (controllers.IPPORollout, SURVEY §8 row f2) against the reference's roll_out loop
(controller/ippo/IPPO.py:128-210) written on the single-environment façade.  CPU: through the host emulation of the
engine (tests/emu, test infrastructure); -m gpu: through the CUDA library."""
import os
import subprocess

import numpy as np
import pytest

from tests import helpers
import torch

from multi_agent_rl_wrsn_b200 import _lib, synthetic
from multi_agent_rl_wrsn_b200.controllers import select_batch
from oracle.ref_runner import reference_root
from tests import parity_cases as pc
from tests.helpers import REPO

EMU_DIR = os.path.join(REPO, "tests", "emu")


@pytest.fixture()
def emu_library():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)
    helpers.use_host_build()
    yield
    helpers.use_cuda_build_lazy()


def _scenarios():
    return [synthetic(num_nodes=40, num_targets=120, seed=s, num_gateways=2) for s in (3, 4)]


def test_ippo_rollout_equals_reference_loop_emu(emu_library):
    n_tr, episodes = pc.check_ippo_rollout(_scenarios(), "cpu", num_envs=4, steps=70, with_obs=False)
    assert n_tr > 200 and episodes >= 2


def test_ippo_rollout_with_observations_emu(emu_library):
    """The same with the observation record (prev_state / state of every transition) and a critic that looks at the maps."""
    n_tr, episodes = pc.check_ippo_rollout(_scenarios(), "cpu", num_envs=3, steps=40, with_obs=True)
    assert n_tr > 80


@pytest.mark.parametrize("with_obs", [False, True])
def test_windows_with_open_decisions_lose_nothing(emu_library, with_obs):
    """keep_open: the same 60 steps collected in 5 windows of 12 give the transitions of the reference's loop, all of them, in order
    (decisions still open at a window end are saved and linked from the next window; episode ends clear them)."""
    n_tr, episodes = pc.check_ippo_rollout(_scenarios(), "cpu", num_envs=3, steps=60, with_obs=with_obs, windows=5)
    assert n_tr > 100 and episodes >= 1


def test_windows_carry_over(emu_library):
    """A record is reused window after window: carry_over on a fresh record changes nothing; after a window it starts from
    the open requests and drops the links into the finished window."""
    from multi_agent_rl_wrsn_b200 import BatchedWRSN
    from multi_agent_rl_wrsn_b200.controllers import IPPORollout
    env = BatchedWRSN(_scenarios(), num_agent=3, num_envs=4, device="cpu")
    ro = IPPORollout(env, 12, action_shape=(3,), with_obs=False)            # resets the never-reset environments itself
    first = ro.agent[0].clone()
    assert bool((first >= 0).all())
    ro.carry_over()
    assert torch.equal(ro.agent[0], first)
    pol = pc._toy_policy(np.arange(4), lambda: env.req.now, False)
    ro.collect(pol)
    n1 = sum(int(ro.transitions(i)[0].numel()) for i in range(3))
    last_agent, last_now = ro.agent[12].clone(), ro.now[12].clone()
    ro.carry_over()
    assert torch.equal(ro.agent[0], last_agent) and torch.equal(ro.now[0], last_now)
    assert int((ro.link >= 0).sum()) == 0 and int((ro.last >= 0).sum()) == 0
    ro.collect(pol)
    n2 = sum(int(ro.transitions(i)[0].numel()) for i in range(3))
    assert n1 > 0 and n2 > 0
    for i in range(3):
        t, b, tp = ro.transitions(i)
        assert bool((tp < t).all()) and bool((ro.agent[tp, b] == i).all()) and bool((ro.agent[t, b] == i).all())


@pytest.mark.gpu
def test_ippo_rollout_equals_reference_loop_gpu():
    n_tr, episodes = pc.check_ippo_rollout(_scenarios(), "cuda", num_envs=6, steps=90)
    assert n_tr > 400 and episodes >= 2


def test_select_batch():
    """IPPO.py:193-200: the half with the most unusual rewards, the rest drawn from the first len - half indices."""
    g = torch.Generator().manual_seed(0)
    r = torch.randn(300, generator=g)
    idx = select_batch(r, 64, generator=g)
    assert idx.shape == (64,)
    top = np.argsort(np.abs(r.numpy() - r.numpy().mean()), kind="stable")[-32:]
    assert np.array_equal(idx[:32].numpy(), top)
    rest = idx[32:].numpy()
    assert len(set(rest.tolist())) == 32 and rest.max() < 300 - 32 and rest.min() >= 0
    with pytest.raises(ValueError):
        select_batch(torch.zeros(40), 64)


class _TinyActor(torch.nn.Module):
    """Same interface as the reference's UNet actor (controller/ppo/actor/UnetActor.py:73-80): (mean, log_std) maps, squeezed."""

    def __init__(self, seed, size):
        super().__init__()
        torch.manual_seed(seed)
        self.conv = torch.nn.Conv2d(4, 1, kernel_size=3, padding=1)
        self.log_std = torch.nn.Parameter(torch.full((1, 1, size, size), -1.0 - 0.1 * seed))

    def forward(self, x):
        mean = self.conv(x)
        return mean.squeeze(), self.log_std.expand_as(mean).squeeze()


def test_per_agent_policy_matches_ippo_evaluate():
    """The stored log-probability is what IPPO.evaluate (IPPO.py:108-115) recomputes with the same actor for the stored
    action, request by request, and every request went to its own agent's actor (also for a group of one)."""
    from torch.distributions.normal import Normal
    from multi_agent_rl_wrsn_b200.controllers import PerAgentPolicy
    S, B = 12, 9
    actors = [_TinyActor(s, S) for s in range(3)]
    g = torch.Generator().manual_seed(5)
    obs = torch.rand((B, 4, S, S), generator=g)
    agent = torch.tensor([0, 2, 2, 0, 0, 2, 0, 1, 2], dtype=torch.int32)           # agent 1: a group of one
    x, lp = PerAgentPolicy(actors, generator=g)(agent, obs)
    assert x.shape == (B, S, S) and lp.shape == (B,)
    for b in range(B):
        with torch.no_grad():
            mean, log_std = actors[int(agent[b])](obs[b:b + 1])
        ref = Normal(mean, log_std.exp()).log_prob(x[b]).sum().detach()
        assert abs(float(ref) - float(lp[b])) <= 1e-4 * max(1.0, abs(float(ref))), b
        with torch.no_grad():
            m2, ls2 = actors[(int(agent[b]) + 1) % 3](obs[b:b + 1])
        other = Normal(m2, ls2.exp()).log_prob(x[b]).sum().detach()
        assert abs(float(other) - float(lp[b])) > 1e-3
    with pytest.raises(ValueError):
        PerAgentPolicy(actors[:2])(agent, obs)


REFERENCE = reference_root()


@pytest.mark.skipif(REFERENCE is None, reason="needs a checkout of the reference (set WRSN_REFERENCE_ROOT)")
def test_reference_networks_fit_the_batched_interfaces():
    """The reference's own UNet actor and CNNCritic (imported unmodified, CPU) behind PerAgentPolicy and ppo_update: shapes,
    the squeezed batch of one, and log-probabilities that IPPO.evaluate reproduces."""
    import sys
    from torch.distributions.normal import Normal
    from multi_agent_rl_wrsn_b200.controllers import PerAgentPolicy, ppo_update
    shims = os.path.join(REPO, "oracle", "shims")                          # matplotlib / gym stand-ins (the image has neither)
    sys.path[:0] = [REFERENCE, shims]
    loaded = set(sys.modules)
    try:
        from controller.ppo.actor.UnetActor import UNet
        from controller.ppo.critic.CNNCritic import CNNCritic
    finally:
        sys.path.remove(REFERENCE)
        sys.path.remove(shims)
        for name in set(sys.modules) - loaded:                             # leave no reference / shim modules behind
            if name.split(".")[0] in ("controller", "utils", "matplotlib", "gym", "seaborn", "simpy"):
                del sys.modules[name]
    torch.manual_seed(0)
    actors, critics = [UNet(), UNet()], [CNNCritic(), CNNCritic()]
    obs = torch.rand((5, 4, 100, 100))
    agent = torch.tensor([0, 0, 1, 0, 0], dtype=torch.int32)              # agent 1: a batch of one (UNet squeezes it away)
    x, lp = PerAgentPolicy(actors)(agent, obs)
    assert x.shape == (5, 100, 100) and lp.shape == (5,)
    with torch.no_grad():
        mean, log_std = actors[0](obs[[0, 1, 3, 4]])
        ref = Normal(mean, log_std.exp()).log_prob(x[[0, 1, 3, 4]]).sum((1, 2))          # IPPO.evaluate :108-115
    assert torch.allclose(ref, lp[[0, 1, 3, 4]], rtol=1e-4)
    values = critics[0](obs).sum(1)                                         # IPPO.get_value :117-119
    assert values.shape == (5,)
    idx = torch.tensor([0, 1, 3, 4])
    batch = dict(states=obs[idx], actions=x[idx], log_probs=lp[idx], advantages=torch.randn(4), returns=torch.randn(4),
                 values=values[idx].detach())
    args = dict(clip=0.2, n_updates_per_iteration=1, norm_adv=True, minibatch_size=4, ent_coef=0.0, vf_coef=0.5,
                max_grad_norm=0.5, clip_vloss=True)
    opt = torch.optim.Adam(list(actors[0].parameters()) + list(critics[0].parameters()), lr=3e-4)
    before = actors[0].out_mean.conv.weight.detach().clone()
    st = ppo_update(actors[0], critics[0], opt, batch, args)
    assert torch.isfinite(st["loss"]) and abs(float(st["approx_kl"])) < 1e-3    # same parameters: ratio = 1 at the first minibatch
    assert not torch.equal(before, actors[0].out_mean.conv.weight.detach())
