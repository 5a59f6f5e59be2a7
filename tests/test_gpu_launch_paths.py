"""The two forms of the pipelined learner step (sacb_per_step: one captured graph in staged mode, the same launches enqueued directly in
persistent mode) against the three calls it stands for: a frame counter set between steps, and the kernel launches they count."""
import numpy as np
import pytest
import torch

from tests.golden import cases
from tests.util import NETS, make_agent

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def per_agents(hw, launch, n=3000, cap=4096):
    """Two tiny_m2 agents over the same prioritized buffer contents (IS-weighted losses: beta reaches the weights)."""
    case = cases.UPDATE_CASES["tiny_m2"]
    rng = np.random.RandomState(5)
    S, A = rng.standard_normal((n, case["obs"])).astype(np.float32), rng.uniform(-0.4, 0.4, (n, case["act"])).astype(np.float32)
    R, S2, D = rng.standard_normal(n).astype(np.float32), rng.standard_normal((n, case["obs"])).astype(np.float32), (rng.uniform(size=n) < 0.1)
    pri = np.zeros(cap, np.float32)
    pri[:n] = np.abs(rng.standard_normal(n)) + 1e-6
    agents = []
    for _ in range(2):
        agent, _st = make_agent(hw, case, math="bf16x3", launch=launch, capacity=cap, replay="per", per_weighted_loss=True)
        agent.replay_buffer.push_many(S, A, R, S2, D)
        agent.replay_buffer.set_priorities(pri)
        agents.append(agent)
    return case["batch"], cap, agents


def sequential_step(hw, agent, B):
    N, lib = hw._native, hw._native.lib()
    N.check(lib.sacb_per_sample(agent._h, 0, None, B, None, None, None, None, None, None, None))
    N.check(lib.sacb_update(agent._h, B, None, None, None, None, N.USE_LAST_SAMPLE | N.NO_LOSS_READBACK))
    N.check(lib.sacb_per_update_from_td(agent._h, 0, B))


def launches(agent):
    return agent.stats()["kernel_launches"]


@pytest.mark.parametrize("launch", ["staged", "persistent"])
def test_frame_set_between_pipelined_steps(hw, launch):
    """replay_buffer.frame = X between two learner steps reaches the sample the next step enqueues (beta and the uniform draws are keyed
    by the frame counter), whether that step replays the cached step graph or launches directly."""
    N, lib = hw._native, hw._native.lib()
    B, cap, (seq, pipe) = per_agents(hw, launch)
    frame = 60000
    for step in range(7):
        if step == 4:
            seq.replay_buffer.frame = frame
        sequential_step(hw, seq, B)
    for call in range(7):
        if call == 3:      # call i updates on step i's minibatch and draws step i + 1's
            pipe.replay_buffer.frame = frame
        pipe.learner_step(B)
    seq.synchronize(); pipe.synchronize()
    assert seq.replay_buffer.frame == frame + 3 and pipe.replay_buffer.frame == frame + 4      # pipe has drawn step 7's minibatch too
    for net in NETS:
        a, b = getattr(seq, net).state_dict(), getattr(pipe, net).state_dict()
        for k in a:
            assert torch.equal(a[k], b[k]), (net, k)
    pa, pb = np.empty(cap, np.float32), np.empty(cap, np.float32)
    N.check(lib.sacb_per_get_priorities(seq._h, 0, N.ptr(pa), cap))
    N.check(lib.sacb_per_get_priorities(pipe._h, 0, N.ptr(pb), cap))
    assert np.array_equal(pa, pb)
    la, lb = np.zeros(3, np.float32), np.zeros(3, np.float32)
    N.check(lib.sacb_get_losses(seq._h, 0, N.ptr(la))); N.check(lib.sacb_get_losses(pipe._h, 0, N.ptr(lb)))
    assert np.array_equal(la, lb) and np.all(np.isfinite(la))


@pytest.mark.parametrize("launch", ["staged", "persistent"])
def test_pipelined_step_counts_the_launches_of_the_three_calls(hw, launch):
    """kernel_launches of one steady-state sacb_per_step == sacb_per_sample + sacb_update(USE_LAST_SAMPLE) + sacb_per_update_from_td
    (three sampler kernels, the update, write-back and priority maximum); sacb_update_steps(K) counts K steps."""
    N, lib = hw._native, hw._native.lib()
    B, _cap, (seq, pipe) = per_agents(hw, launch)
    for _ in range(2):      # programs built, shadows resident, step graph captured
        sequential_step(hw, seq, B)
        N.check(lib.sacb_per_step(pipe._h, B, None, N.NO_LOSS_READBACK))
    n0 = launches(seq)
    sequential_step(hw, seq, B)
    per_three_calls = launches(seq) - n0
    n0 = launches(pipe)
    N.check(lib.sacb_per_step(pipe._h, B, None, N.NO_LOSS_READBACK))
    per_step = launches(pipe) - n0
    assert per_step == per_three_calls, (per_step, per_three_calls)
    if launch == "persistent":
        assert per_step == 6      # one cooperative launch + 5 replay kernels
    K = 4
    n0 = launches(pipe)
    N.check(lib.sacb_update_steps(pipe._h, B, K, None, N.NO_LOSS_READBACK))
    assert launches(pipe) - n0 == K * per_step
    seq.synchronize(); pipe.synchronize()
