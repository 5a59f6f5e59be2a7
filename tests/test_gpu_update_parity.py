"""GPU parity of SAC.update_parameters (reference sac_imp.py:74-144) through the C ABI.

Chain of evidence: live reference --(tests/golden/*.npz)--> numpy oracle (test_oracle_update_golden.py)
and here: CUDA path vs the oracle on the same seeded inputs AND vs the golden vectors directly.
Tolerances (relative; the north star asks for 1e-3).  Both modes read the SAME bf16 hi/lo pair operands
(2^-17 relative storage rounding of activations / weight shadows; master weights, Adam state, accumulators fp32):
  fp32   (FFMA tile, fp32 products)                          3e-4
  bf16x3 (TMA + tcgen05, 3 MMAs per product, DEFAULT)        3e-4
"""
import os

import numpy as np
import pytest

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.util import PARITY_TOL as TOL
from tests.util import batch_of, grad_close, make_agent, net_params, relerr, relu_hint

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")

CASES = [c for c in cases.UPDATE_CASES if not cases.UPDATE_CASES[c].get("loose")]


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def run_case(hw, name, math, launch):
    case = cases.UPDATE_CASES[name]
    tol = TOL[math]
    g = np.load(os.path.join(GOLD, f"update_{name}.npz"))
    agent, st = make_agent(hw, case, math=math, launch=launch)
    for step in range(case["steps"]):
        b = batch_of(case, step)
        got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=True)
        # ReLU masks: the oracle keeps its own mask wherever |z| >= 1e-4 rms(z) and there the device must agree exactly
        hint = relu_hint(agent, case)
        ref_losses, aux = O.update_parameters(st, b, return_aux=True, relu_hint=hint)
        assert hint.mismatch == 0, (step, hint.mismatch, hint.adopted, hint.ambiguous)
        assert hint.adopted <= 64, (hint.adopted, hint.ambiguous)       # a handful of genuine ties per update, not a drift
        for k in ("q1_loss", "q2_loss", "policy_loss"):
            assert abs(got[k] - ref_losses[k]) <= tol["loss"] * abs(ref_losses[k]) + 1e-6, (step, k, got[k], ref_losses[k])
        # golden (live reference) losses as well
        np.testing.assert_allclose([got["q1_loss"], got["q2_loss"], got["policy_loss"]], g["losses"][step], rtol=2 * tol["loss"], atol=1e-6)
        for net in ("q1", "q2", "policy"):
            gg = agent.exported_grads(net)
            for nm, ref in aux[f"{net}_grads"].items():
                ok, overall, bad = grad_close(gg[nm], ref, tol["grad"], max_flips=0)
                assert ok, (step, net, nm, overall, bad)
                if step == 0:
                    gold = g[f"gradsum/{net}/{nm}"]
                    assert abs(np.linalg.norm(gg[nm].astype(np.float64)) - gold[1]) <= 2 * tol["grad"] * gold[1] + 1e-12
        a = agent.alpha
        a = float(a) if not hasattr(a, "item") else float(a.item())
        assert abs(a - st.alpha) <= 1e-5 * abs(st.alpha), (a, st.alpha)
        np.testing.assert_allclose(a, g["alphas"][step], rtol=2e-5)
    # post-update state: Adam moves every weight by ~lr per step whatever |g| is -> compare in units of lr
    budget = tol["budget"] * st.lr * case["steps"] + 1e-7
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        mine = net_params(agent, net)
        for nm, ref in getattr(st, net).items():
            frac_bad = np.mean(np.abs(mine[nm] - ref) > budget)
            assert frac_bad < tol["frac"], (net, nm, frac_bad, np.abs(mine[nm] - ref).max())
            # directly against the live reference's weights (no oracle, no ReLU hint in between): the oracle<->golden budget
            # (0.02 lr per step) plus the device<->oracle budget; a ReLU tie that falls the other way moves single entries by up to
            # 2 lr (and a weight row fed by that unit by a fraction of lr): the median of the 64 kept values must meet the budget and at
            # most 2 may be off by more than a quarter step -- a wrong-sign or missing step fails on every entry
            dg = np.abs(mine[nm].ravel()[:64] - g[f"paramhead/{net}/{nm}"])
            assert dg.max() < 2.1 * st.lr * case["steps"], (net, nm, dg.max())
            assert np.median(dg) < 2 * budget, (net, nm, np.median(dg), budget)
            assert int(np.sum(dg > 0.25 * st.lr * case["steps"])) <= 2, (net, nm, np.sort(dg)[-4:], budget)
    for net, opt in (("policy", st.policy_opt), ("q1", st.q1_opt), ("q2", st.q2_opt)):
        sd = getattr(agent, f"{net}_optimizer").state_dict()
        names = list(getattr(st, net).keys())
        for i, nm in enumerate(names):
            assert int(sd["state"][i]["step"]) == case["steps"]
            assert grad_close(sd["state"][i]["exp_avg"].cpu().numpy(), opt.m[nm], tol["adam"], max_flips=0)[0], (net, nm)
            assert grad_close(sd["state"][i]["exp_avg_sq"].cpu().numpy(), opt.v[nm], 2 * tol["adam"], max_flips=0)[0], (net, nm)
    return agent


@pytest.mark.parametrize("name", CASES)
def test_update_fp32_staged(hw, name):
    run_case(hw, name, "fp32", "staged")


@pytest.mark.parametrize("name", CASES)
def test_update_bf16x3_staged(hw, name):
    run_case(hw, name, "bf16x3", "staged")


@pytest.mark.parametrize("name", ["tiny_m2", "c1_bipedal_m1", "c2_humanoid_m2"])
@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
def test_update_persistent_single_launch(hw, name, math):
    """ONE cooperative launch per step (grid barriers between stages) gives the same step as the staged graph."""
    agent = run_case(hw, name, math, "persistent")
    assert agent.stats()["n_stages"] >= 17


def test_persistent_equals_staged_bitwise(hw):
    case = cases.UPDATE_CASES["c1_bipedal_m1"]
    outs = []
    for launch in ("staged", "persistent"):
        agent, _ = make_agent(hw, case, math="fp32", launch=launch)
        for step in range(2):
            b = batch_of(case, step)
            agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
        outs.append({n: net_params(agent, n) for n in ("policy", "q1", "q2_target")})
    for n in outs[0]:
        for k in outs[0][n]:
            np.testing.assert_array_equal(outs[0][n][k], outs[1][n][k])


def test_saturated_case_loose(hw):
    """|x_t| up to ~20: the reference's own fp32 result moves by 1e-2 with a 1-ulp change of tanh (oracle header)."""
    case = cases.UPDATE_CASES["humanoid_m1_saturated"]
    g = np.load(os.path.join(GOLD, "update_humanoid_m1_saturated.npz"))
    agent, st = make_agent(hw, case, math="fp32")
    b = batch_of(case, 0)
    got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    np.testing.assert_allclose([got["q1_loss"], got["q2_loss"], got["policy_loss"]], g["losses"][0], rtol=2e-2)


def test_per_weighted_loss_extension(hw):
    """IS-weighted critic loss (extension H10) against the oracle's per_weights path."""
    case = cases.UPDATE_CASES["tiny_m2"]
    agent, st = make_agent(hw, case, math="fp32")
    b = batch_of(case, 0)
    w = np.random.RandomState(5).uniform(0.2, 1.0, case["batch"]).astype(np.float32)
    ref = O.update_parameters(st, b, per_weights=w)
    got, td = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), is_weights=w, want_td=True)
    for k in ref:
        assert abs(got[k] - ref[k]) <= 2e-4 * abs(ref[k]) + 1e-6
    assert td.shape == (case["batch"],) and np.all(td >= 0)


def test_device_eps_mode_runs_and_learns(hw):
    """Production mode: eps drawn on the device (Philox); losses finite, critic loss decreases on a fixed batch."""
    case = cases.UPDATE_CASES["c1_bipedal_m1"]
    agent, _ = make_agent(hw, case, math="bf16x3")
    b = batch_of(case, 0)
    l0 = agent.update_from_batch(b)
    for _ in range(30):
        l1 = agent.update_from_batch(b)
    assert np.isfinite(list(l1.values())).all()
    assert l1["q1_loss"] < l0["q1_loss"]


@pytest.mark.parametrize("B", [2048])
def test_large_batch_update_matches_oracle(hw, B):
    """BASELINE.json configs[3] in miniature (one rank's share of a large global batch, C2 nets): stages with many more tiles than
    SMs run one resident CTA per SM looping over tiles -- same arithmetic, checked against the oracle (losses, every gradient, alpha)."""
    case = dict(cases.UPDATE_CASES["c2_humanoid_m2"], batch=B, steps=1, seed=77)
    tol = TOL["bf16x3"]
    agent, st = make_agent(hw, case, math="bf16x3")
    b = batch_of(case, 0)
    got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=True)
    hint = relu_hint(agent, case)
    ref_losses, aux = O.update_parameters(st, b, return_aux=True, relu_hint=hint)
    assert hint.mismatch == 0, (hint.mismatch, hint.adopted, hint.ambiguous)
    for k in ("q1_loss", "q2_loss", "policy_loss"):
        assert abs(got[k] - ref_losses[k]) <= tol["loss"] * abs(ref_losses[k]) + 1e-6, (k, got[k], ref_losses[k])
    for net in ("q1", "q2", "policy"):
        gg = agent.exported_grads(net)
        for nm, ref in aux[f"{net}_grads"].items():
            ok, overall, bad = grad_close(gg[nm], ref, tol["grad"], max_flips=0)
            assert ok, (net, nm, overall, bad)
    a = agent.alpha
    a = float(a) if not hasattr(a, "item") else float(a.item())
    assert abs(a - st.alpha) <= 1e-5 * abs(st.alpha), (a, st.alpha)
    assert agent.stats()["grid"] > 2 * agent.stats()["sm_count"]      # the widest stage really exceeds two waves (tile-loop CTAs)


def test_wide_stream_tiles_equal_128_wide_tiles_bitwise(hw, monkeypatch):
    """Throughput form at B = 8192 (C2 nets): the program built with 128 x 256 stream tiles (two ring slots, four epilogue passes)
    must equal the one built with 128 x 128 tiles bit for bit -- same K order and the same three products per output element."""
    case = dict(cases.UPDATE_CASES["c2_humanoid_m2"], batch=8192, steps=2, seed=78)
    agents = []
    for n256 in ("0", "1"):
        monkeypatch.setenv("SACB_STREAM_N256_MIN", n256)      # read when the update program is built (first update of the handle)
        agent, _ = make_agent(hw, case, math="bf16x3")
        losses = []
        for step in range(case["steps"]):
            b = batch_of(case, step)
            losses.append(agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"])))
        agents.append((agent, losses))
    (a0, l0), (a1, l1) = agents
    assert a1.stats()["n_tiles"] < a0.stats()["n_tiles"]      # the second program really is cut into wider (fewer) tiles
    assert l0 == l1, (l0, l1)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        p0, p1 = net_params(a0, net), net_params(a1, net)
        for nm in p0:
            np.testing.assert_array_equal(p0[nm], p1[nm], err_msg=f"{net}.{nm}")
    assert np.isfinite(list(l1[-1].values())).all()


ODD_SHAPES = {
    "wide_action_m1": dict(obs=20, act=40, hidden=64, n_hidden=2, batch=37, steps=2, seed=91, bias_scale=0.05, head_scale=0.25),     # 2A = 80 > one 64-column tile
    "one_action_m2": dict(obs=7, act=1, hidden=8, n_hidden=3, batch=5, steps=2, seed=92, bias_scale=0.05),                           # everything smaller than a tile
    "odd_everything_m2": dict(obs=131, act=9, hidden=72, n_hidden=3, batch=129, steps=1, seed=93, bias_scale=0.05, head_scale=0.5),  # no dimension a multiple of 64
}


@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
@pytest.mark.parametrize("name", list(ODD_SHAPES))
def test_odd_shapes_match_oracle(hw, name, math):
    """Ragged tiles everywhere (TMA zero fill, partial Adam tiles, heads wider than one tile, B below / just above a tile)."""
    case = ODD_SHAPES[name]
    tol = TOL[math]
    agent, st = make_agent(hw, case, math=math)
    for step in range(case["steps"]):
        b = batch_of(case, step)
        got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=True)
        hint = relu_hint(agent, case)
        ref_losses, aux = O.update_parameters(st, b, return_aux=True, relu_hint=hint)
        assert hint.mismatch == 0, (step, hint.mismatch, hint.adopted, hint.ambiguous)
        for k in ("q1_loss", "q2_loss", "policy_loss"):
            assert abs(got[k] - ref_losses[k]) <= tol["loss"] * abs(ref_losses[k]) + 1e-6, (step, k, got[k], ref_losses[k])
        for net in ("q1", "q2", "policy"):
            gg = agent.exported_grads(net)
            for nm, ref in aux[f"{net}_grads"].items():
                ok, overall, bad = grad_close(gg[nm], ref, tol["grad"], max_flips=0)
                assert ok, (step, net, nm, overall, bad)
    budget = tol["budget"] * st.lr * case["steps"] + 1e-7
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        mine = net_params(agent, net)
        for nm, ref in getattr(st, net).items():
            assert np.mean(np.abs(mine[nm] - ref) > budget) < tol["frac"], (net, nm)
