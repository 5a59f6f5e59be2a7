"""GPU tests of (a) the networks as callables -- QNetwork.forward, GaussianPolicy.forward / .sample through sacb_q_forward,
sacb_policy_forward, sacb_policy_sample -- and (b) checkpoint interop with files the REFERENCE wrote: its shipped
results/*/best_model.pt (obs 24 and obs 376) and a save() / save_checkpoint() pair written by the live reference
(tests/golden/make_golden.py ckpt), (c) the resident weight shadows (no re-shadow stage) against the re-derive-every-step form."""
import os

import numpy as np
import pytest
import torch

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.util import batch_of, make_agent, net_params, state_from_checkpoint

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
SHIPPED = {"bipedal": dict(obs=24, act=4, hidden=256, n_hidden=2, batch=256, seed=31),
           "humanoid376": dict(obs=376, act=17, hidden=256, n_hidden=2, batch=256, seed=32)}


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


@pytest.mark.parametrize("name", cases.NETS_CASES)
def test_network_callables_match_reference(hw, name):
    """networks_model1.py:27-33, :65-99 / networks_model2.py:37-46, :85-120 on 32 rows: library vs oracle vs live-reference golden."""
    case = cases.UPDATE_CASES[name]
    g = np.load(os.path.join(GOLD, f"nets_{name}.npz"))
    agent, st = make_agent(hw, case, math="fp32")
    inp = cases.nets_inputs(case, 32)
    q1 = agent.q1(torch.from_numpy(inp["s"]), torch.from_numpy(inp["a"])).numpy()
    q2t = agent.q2_target(inp["s"], inp["a"]).numpy()
    assert q1.shape == (32, 1)
    np.testing.assert_allclose(q1, O.q_forward(st.q1, inp["s"], inp["a"], st.n_hidden), rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(q1, g["q1"], rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(q2t, g["q2_target"], rtol=2e-5, atol=5e-6)
    mean, log_std = agent.policy(torch.from_numpy(inp["s"]))
    np.testing.assert_allclose(mean.numpy(), g["mean"], rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(log_std.numpy(), g["log_std"], rtol=2e-5, atol=5e-6)
    action, logp = agent.policy.sample(torch.from_numpy(inp["s"]), eps=inp["eps"])
    assert action.shape == (32, case["act"]) and logp.shape == (32, 1)
    ref_a, ref_lp = O.policy_sample(st.policy, inp["s"], inp["eps"], st.n_hidden, st.action_scale, st.action_bias)
    np.testing.assert_allclose(action.numpy(), ref_a, rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(logp.numpy(), ref_lp, rtol=1e-4, atol=2e-4)
    np.testing.assert_allclose(action.numpy(), g["action"], rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(logp.numpy(), g["log_prob"], rtol=1e-4, atol=2e-4)
    a2, lp2 = agent.policy.sample(inp["s"])                      # production draw (Philox): inside the bounds, finite log-prob
    assert np.all(np.abs(a2.numpy()) <= 0.4 + 1e-6) and np.isfinite(lp2.numpy()).all()
    a3, _ = agent.policy.sample(inp["s"])
    assert not np.array_equal(a2.numpy(), a3.numpy())              # the counter advances: a new draw every call


def test_uniform_sample_any_size(hw):
    """ReplayBuffer.sample (replay_buffer.py:13-19) through sacb_sample_uniform, batch far above the handle's max_batch."""
    buf = hw.ReplayBuffer(10000)
    n = 6000
    for i in range(n):
        buf.push(np.full(3, i, np.float32), np.full(2, -i, np.float32), float(i), np.full(3, i + 0.5, np.float32), i % 5 == 0)
    import random
    random.seed(5)
    s, a, r, s2, d = buf.sample(5000)
    random.seed(5)
    picks = np.asarray(random.sample(range(n), 5000))
    np.testing.assert_array_equal(r, picks.astype(np.float32))
    np.testing.assert_array_equal(s[:, 0], r)
    np.testing.assert_array_equal(s2[:, 2], r + 0.5)
    np.testing.assert_array_equal(d, (picks % 5 == 0).astype(np.float32))
    assert len(buf.buffer) == n


@pytest.mark.parametrize("tag", list(SHIPPED))
def test_load_shipped_reference_checkpoints(hw, tag):
    """SAC.load (sac_imp.py:164-173) of the reference's own shipped best_model.pt: acting, Q values and one seeded update
    reproduce what the live reference computed from the same file (tests/golden/shipped_*_expected.npz)."""
    case = SHIPPED[tag]
    exp = np.load(os.path.join(GOLD, f"shipped_{tag}_expected.npz"))
    path = os.path.join(GOLD, f"shipped_{tag}_best_model.pt")
    hw.use_networks("model1")
    agent = hw.SAC(case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", math="bf16x3", max_batch=case["batch"], capacity=1024)
    agent.load(path)
    st, ck = state_from_checkpoint(path, case)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        for k, v in net_params(agent, net).items():
            np.testing.assert_array_equal(v, ck[f"{net}_state_dict"][k].cpu().numpy())
    a = agent.alpha
    assert torch.is_tensor(a) and abs(float(a) - float(exp["alpha_loaded"])) < 1e-7     # the file holds a tensor (sac_imp.py:135)
    obs_mat = np.random.RandomState(77 + case["seed"]).standard_normal((8, case["obs"])).astype(np.float32)
    got = np.stack([agent.select_action(o, evaluate=True) for o in obs_mat])
    np.testing.assert_allclose(got, exp["select_eval"], rtol=1e-4, atol=1e-5)
    inp = cases.nets_inputs(case, 16)
    np.testing.assert_allclose(agent.q1(inp["s"], inp["a"]).numpy(), exp["q1"], rtol=1e-4, atol=1e-4)
    b = O.make_batch(case["obs"], case["act"], case["batch"], seed=case["seed"] * 100)
    l = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    ref = O.update_parameters(st, b)
    np.testing.assert_allclose([l["q1_loss"], l["q2_loss"]], exp["losses"][0][:2], rtol=1e-3)
    np.testing.assert_allclose([l["q1_loss"], l["q2_loss"]], [ref["q1_loss"], ref["q2_loss"]], rtol=3e-4)
    np.testing.assert_allclose(l["policy_loss"], exp["losses"][0][2], rtol=5e-3)        # trained heads saturate tanh on N(0,1) observations
    np.testing.assert_allclose(float(agent.alpha), exp["alpha_after"], rtol=1e-5)


def test_resume_checkpoint_written_by_the_reference(hw):
    """load() / load_checkpoint() (sac_imp.py:164-173, :203-233) of files the live reference wrote after two updates: weights,
    Adam state, log_alpha, deque contents -- and the NEXT update reproduces the reference's own third step within 3e-4."""
    case = cases.UPDATE_CASES["tiny_m1"]
    exp = np.load(os.path.join(GOLD, "ckpt_ref_expected.npz"))
    p_ck, p_save = os.path.join(GOLD, "ckpt_ref_checkpoint.pt"), os.path.join(GOLD, "ckpt_ref_save.pt")
    hw.use_networks("model1")
    agent = hw.SAC(case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", math="fp32", max_batch=case["batch"], capacity=256)
    ep, steps = agent.load_checkpoint(p_ck)
    assert (ep, steps) == (7, 123)
    ck = torch.load(p_ck, map_location="cpu", weights_only=False)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        for k, v in net_params(agent, net).items():
            np.testing.assert_array_equal(v, ck[f"{net}_state_dict"][k].numpy())
    osd = agent.q1_optimizer.state_dict()
    assert float(osd["state"][0]["step"]) == 2.0
    np.testing.assert_array_equal(osd["state"][2]["exp_avg_sq"].cpu().numpy(), ck["q1_optimizer_state_dict"]["state"][2]["exp_avg_sq"].numpy())
    assert abs(float(agent.log_alpha) - float(ck["log_alpha"])) < 1e-9
    stored = agent.replay_buffer.buffer
    want = cases.ckpt_transitions(case)
    assert len(stored) == len(want) == 20
    for got_t, ref_t in zip(stored, want):
        np.testing.assert_array_equal(got_t[0], ref_t[0].astype(np.float32))
        np.testing.assert_array_equal(got_t[1], ref_t[1])
        assert got_t[2] == np.float32(ref_t[2]) and got_t[4] == ref_t[4]
    b = batch_of(case, 2)
    l = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    np.testing.assert_allclose([l["q1_loss"], l["q2_loss"], l["policy_loss"]], exp["next_losses"][0], rtol=3e-4)
    np.testing.assert_allclose(float(agent.alpha), exp["next_alpha"], rtol=1e-5)
    obs_vec = np.random.RandomState(77 + case["seed"]).standard_normal(case["obs"]).astype(np.float32)
    np.testing.assert_allclose(agent.select_action(obs_vec, evaluate=True), exp["select_eval_after"], rtol=1e-3, atol=2e-5)
    other = hw.SAC(case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", math="fp32", max_batch=case["batch"], capacity=256)
    other.load(p_save)
    sv = torch.load(p_save, map_location="cpu", weights_only=False)
    np.testing.assert_array_equal(net_params(other, "policy")["mean.weight"], sv["policy_state_dict"]["mean.weight"].numpy())
    assert abs(float(other.alpha) - float(sv["alpha"])) < 1e-9


def test_write_product_checkpoints_for_the_reference(hw, tmp_path):
    """Writes save() / save_checkpoint() files from the product after two seeded updates, then takes the next step.  The files
    and that step are what tests/golden/product_*.pt and product_expected.npz hold (written by this test on a B200), which the
    CPU-side test (tests/test_cabi.py::test_reference_loads_product_checkpoints) checks against the reference's load code."""
    case = cases.UPDATE_CASES["tiny_m1"]
    agent, st = make_agent(hw, case, math="fp32", capacity=128)
    for step in range(2):
        b = batch_of(case, step)
        agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    for t in cases.ckpt_transitions(case):
        agent.replay_buffer.push(*t)
    out_dir = str(tmp_path)
    agent.save(os.path.join(out_dir, "product_save.pt"))
    agent.save_checkpoint(os.path.join(out_dir, "product_checkpoint.pt"), episode=3, total_steps=45)
    b = batch_of(case, 2)
    l = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    np.savez(os.path.join(out_dir, "product_expected.npz"), next_losses=np.array([l["q1_loss"], l["q2_loss"], l["policy_loss"]]),
             next_alpha=np.array(float(agent.alpha)))
    ck = torch.load(os.path.join(out_dir, "product_checkpoint.pt"), map_location="cpu", weights_only=False)
    assert len(ck["replay_buffer"]) == 20 and float(ck["policy_optimizer_state_dict"]["state"][0]["step"]) == 2.0
    committed = np.load(os.path.join(GOLD, "product_expected.npz"))
    np.testing.assert_allclose([l["q1_loss"], l["q2_loss"], l["policy_loss"]], committed["next_losses"], rtol=3e-4)
    np.testing.assert_allclose(float(agent.alpha), committed["next_alpha"], rtol=1e-5)


def test_resident_shadows_equal_rederived_shadows(hw):
    """The Adam / Polyak epilogues keep the bf16 pair shadows of all five nets current, so the steady-state program has no
    shadow stage.  Bitwise equal to re-deriving every shadow from the fp32 weights before every step (round-1 behaviour)."""
    from humanoid_walking_with_sac_b200 import _native as N
    case = cases.UPDATE_CASES["c1_bipedal_m1"]
    outs = []
    for rederive in (False, True):
        agent, _ = make_agent(hw, case, math="bf16x3")
        for step in range(4):
            b = batch_of(case, step % 3)
            if rederive:
                agent.invalidate_shadows()
            agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
        outs.append({n: net_params(agent, n) for n in ("policy", "q1", "q2", "q1_target", "q2_target")})
        outs[-1]["stages"] = agent.stats()["n_stages"]
    for n in ("policy", "q1", "q2", "q1_target", "q2_target"):
        for k in outs[0][n]:
            np.testing.assert_array_equal(outs[0][n][k], outs[1][n][k])


def test_alias_write_between_updates_is_picked_up(hw):
    """A write through the torch aliases (what load_state_dict does) after the shadows became resident: the next update must see it."""
    case = cases.UPDATE_CASES["tiny_m2"]
    agent, st = make_agent(hw, case, math="fp32")
    for step in range(2):
        b = batch_of(case, step)
        agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
        O.update_parameters(st, b)
    with torch.no_grad():
        agent.q1.fc2.weight.mul_(1.5)
        agent.policy.fc1.weight.add_(0.01)
        agent.q2_target.fc1.weight.mul_(0.5)
    # the oracle follows the DEVICE's current weights (sign ties of the first two steps aside, they agree to ~1e-7)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        setattr(st, net, {k: v.copy() for k, v in net_params(agent, net).items()})
    b = batch_of(case, 2)
    got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]))
    ref = O.update_parameters(st, b)
    for k in ref:
        assert abs(got[k] - ref[k]) <= 3e-4 * abs(ref[k]) + 1e-6, (k, got[k], ref[k])
