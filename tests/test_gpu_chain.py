"""Chained launches of the tensor-core update program (program.cu: find_chains) against the persistent launch, which never chains.

Chaining changes no arithmetic: the staged bf16x3 program (whose row-local MLP layers run as thread-block-cluster launches) and the
single persistent launch must leave bit-identical losses, parameters and Adam moments.  Two updates from a fresh handle: the first
runs the program that re-derives the weight shadows, the second the resident one.
"""
import numpy as np
import pytest

from tests.golden import cases
from tests.util import batch_of, make_agent, net_params

pytestmark = pytest.mark.gpu

NETS = ("policy", "q1", "q2", "q1_target", "q2_target")
CASES = {
    "c2_humanoid_m2": cases.UPDATE_CASES["c2_humanoid_m2"],
    "c3_nao_m2": cases.UPDATE_CASES["c3_nao_m2"],
    "c1_bipedal_m1": cases.UPDATE_CASES["c1_bipedal_m1"],      # H = 256: clusters of 4
    "tiny_m2": cases.UPDATE_CASES["tiny_m2"],                  # H = 48: one-CTA chains
    "c2_humanoid_m2_b200": dict(cases.UPDATE_CASES["c2_humanoid_m2"], batch=200),      # ragged last row block
}


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def _run(hw, case, launch):
    agent, _ = make_agent(hw, case, math="bf16x3", launch=launch)
    losses = []
    for step in range(2):
        b = batch_of(case, step)
        got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
        losses.append([got[k] for k in sorted(got)])
    out = {"losses": np.array(losses, np.float64)}
    for n in NETS:
        for k, v in net_params(agent, n).items():
            out[f"{n}.{k}"] = v
    for opt in ("policy_optimizer", "q1_optimizer", "q2_optimizer"):
        for i, s in getattr(agent, opt).state_dict()["state"].items():
            for k in ("exp_avg", "exp_avg_sq"):
                out[f"{opt}.{i}.{k}"] = np.asarray(s[k].detach().cpu().numpy()).copy()
    return out


@pytest.mark.parametrize("name", list(CASES))
def test_staged_equals_persistent_bitwise(hw, name):
    staged, persistent = _run(hw, CASES[name], "staged"), _run(hw, CASES[name], "persistent")
    assert staged.keys() == persistent.keys()
    for k in staged:
        np.testing.assert_array_equal(staged[k], persistent[k], err_msg=k)


def test_c2_update_is_chained(hw):
    """At C2 the three 3-layer chains (target critics, updated critics, dL/da through both critics) are one launch each: 25 stages, 19
    launches, plus the batch upload of update_from_batch (26 without chains).  The forward chain on [s2; s] and (s, a) needs 16 resident
    clusters of 8 CTAs, one more than a B200 holds, so it keeps its four launches."""
    case = CASES["c2_humanoid_m2"]
    agent, _ = make_agent(hw, case, math="bf16x3")
    b = batch_of(case, 0)
    agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    n0 = agent.stats()["kernel_launches"]
    b = batch_of(case, 1)
    agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    assert agent.stats()["kernel_launches"] - n0 <= 20
