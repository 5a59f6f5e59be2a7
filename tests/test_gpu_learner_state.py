"""The optimizer state and prioritized-buffer accessors that SAC and PopulationSAC share.

1. Loading a checkpoint written before the first update (torch.optim.Adam state_dicts with an empty `state`) leaves what a fresh
   torch Adam holds, step 0 and zero moments, whatever the learner held before: a trained SAC (load_checkpoint) or population member
   (load_agent_checkpoint) then takes the same next step as the agent that wrote the file, bit for bit.
2. set_priorities refuses a p_alpha table of another length than the priorities, on a standalone buffer and on a population member;
   a population member's sample refuses more rows than max_batch."""
import numpy as np
import pytest
import torch

from tests.golden import cases
from tests.test_gpu_population_hparams import Setup
from tests.util import batch_of, make_agent

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    yield hw
    hw.use_networks("model1")


def tensors_of(checkpoint, prefix=""):
    """{key path: array} of every tensor in a checkpoint dictionary (nets, Adam moments and steps, alpha, log_alpha)."""
    out = {}
    for k, v in checkpoint.items():
        if isinstance(v, dict):
            out.update(tensors_of(v, f"{prefix}{k}."))
        elif torch.is_tensor(v):
            out[f"{prefix}{k}"] = v.detach().cpu().numpy()
    return out


def assert_same_tensors(got, want, tag):
    got, want = tensors_of(got), tensors_of(want)
    assert set(got) == set(want), (tag, set(got) ^ set(want))
    for k, v in want.items():
        np.testing.assert_array_equal(got[k], v, err_msg=f"{tag} {k}")


def sac_checkpoint(agent, path):
    agent.save_checkpoint(str(path), 0, 0, replay_buffer=False)
    return torch.load(str(path), map_location="cpu", weights_only=False)


def assert_step0(checkpoint):
    for name in ("policy", "q1", "q2", "alpha"):
        assert checkpoint[f"{name}_optimizer_state_dict"]["state"] == {}, name


@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
def test_sac_resumes_a_step0_checkpoint_like_a_fresh_adam(hw, tmp_path, math):
    """A SAC trained for two updates loads another agent's step-0 checkpoint; its next update equals that agent's first, bitwise."""
    case = cases.UPDATE_CASES["tiny_m1"]
    fresh, _ = make_agent(hw, dict(case, seed=99), math=math)
    assert_step0(sac_checkpoint(fresh, tmp_path / "step0.pt"))
    trained, _ = make_agent(hw, case, math=math)
    for step in range(2):
        b = batch_of(case, step)
        trained.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    trained.load_checkpoint(str(tmp_path / "step0.pt"))
    b = batch_of(case, 2)
    assert trained.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"])) == fresh.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    assert_same_tensors(sac_checkpoint(trained, tmp_path / "trained.pt"), sac_checkpoint(fresh, tmp_path / "fresh.pt"), "SAC")


def test_member_resumes_a_step0_checkpoint_like_a_fresh_adam(hw, tmp_path):
    """Member 1 of a population trained for two updates loads a SAC's step-0 checkpoint; on the same rows and noise its next update
    equals the SAC's first, bitwise (the population's defaults are the SAC's hyperparameters)."""
    S = Setup(hw, "tiny_m2", 2, steps=3)
    pop = S.population({})
    for k in range(2):
        S.step(pop, k)
    fresh = S.single(1, {"lr": 3e-4, "gamma": 0.99, "tau": 0.005, "alpha": 0.2, "target_entropy": -float(S.act)}, seed=55)
    assert_step0(sac_checkpoint(fresh, tmp_path / "step0.pt"))
    pop.load_agent_checkpoint(1, str(tmp_path / "step0.pt"))
    assert S.step(pop, 2)[1] == S.single_step(fresh, 1, 2)
    member = {k: v for k, v in pop.agent_checkpoint(1).items() if k != "sacb_hyperparameters"}
    assert_same_tensors(member, sac_checkpoint(fresh, tmp_path / "fresh.pt"), "member 1")


def test_p_alpha_of_another_length_is_refused(hw):
    buf = hw.PrioritizedReplayBuffer(64)
    buf.push_many(np.zeros((40, 3)), np.zeros((40, 2)), np.zeros(40), np.zeros((40, 3)), np.zeros(40))
    before = buf.priorities
    for n_pa in (9, 11):
        with pytest.raises(ValueError):
            buf.set_priorities(np.ones(10, np.float32), np.ones(n_pa, np.float32))
    np.testing.assert_array_equal(buf.priorities, before)
    pop = hw.PopulationSAC(2, 3, 2, hidden_dim=16, device="cuda", capacity=64, max_batch=16, replay="per")
    pop.push_many(1, np.zeros((40, 3)), np.zeros((40, 2)), np.zeros(40), np.zeros((40, 3)), np.zeros(40))
    before = pop.priorities(1)
    for n_pa in (9, 11):
        with pytest.raises(ValueError):
            pop.set_priorities(1, np.ones(10, np.float32), np.ones(n_pa, np.float32))
    np.testing.assert_array_equal(pop.priorities(1), before)
    with pytest.raises(ValueError):      # more rows than max_batch
        pop.sample(1, 32)
    assert len(pop.sample(1, 16)[5]) == 16
