"""Large-batch programs (BASELINE.json configs[3]) against the oracle: the fused-Adam update of one agent in the throughput form,
and the data-parallel backward whose gradients are exported instead of applied.

Both take the throughput form of the update program (the widest GEMM stage has more than two waves of tiles): stream tiles of
128 rows, mixed stages cut in two, and Adam epilogues that write the policy and Polyak-target shadows from their registers (no
T_SHADOW tasks), so a wrong shadow store first shows in step 2.  A program that exports without applying (data-parallel backward)
also splits every dW GEMM over K into up to 16 chunks, cuts the bias / output-layer column sums into 1024-row chunks once B > 2048,
and accumulates both into the zeroed gradient slab with atomics: those results are compared with tolerances, never bitwise.
Tolerances are those of test_gpu_update_parity (bf16x3)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.test_gpu_update_parity import TOL as PARITY_TOL
from tests.util import batch_of, grad_close, make_agent, net_params, relerr, relu_hint

pytestmark = pytest.mark.gpu
TOL = PARITY_TOL["bf16x3"]
NETS = ("policy", "q1", "q2", "q1_target", "q2_target")
# Data-parallel backward.  SPLIT_TOL: the same gradient summed in another order where every fp32 accumulation chain is short (the
# bound of the GEMM self-tests).  A GEMM accumulates over K in fp32 in tensor memory, and that error grows with the chain: against the
# oracle, the unsplit program's dW at B = K = 2048 / 8192 / 65536 is off by 1.2e-5 / 3e-5 / 3.3e-4, the split one (chains of
# <= 4096 rows) by <= 1e-5 / 1e-5 / 2e-5 (C2, B200).  So the unsplit program is the sharper reference only for short K, and the
# oracle, at SPLIT_ORACLE_TOL, for every B.  A dropped 64-row K block out of 65536 moves a dW by ~3e-2.
SPLIT_TOL = 2e-5
SPLIT_ORACLE_TOL = 4e-5
UNSPLIT_MAX_K = 4096      # batches up to here: the unsplit program's chains are no longer than the split one's


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def case_of(name, B, steps, seed):
    return dict(cases.UPDATE_CASES[name], batch=B, steps=steps, seed=seed)


def alpha_of(agent):
    a = agent.alpha
    return float(a) if not hasattr(a, "item") else float(a.item())


def check_losses(got, ref, tag):
    for k in ("q1_loss", "q2_loss", "policy_loss"):
        assert abs(got[k] - ref[k]) <= TOL["loss"] * abs(ref[k]) + 1e-6, (tag, k, got[k], ref[k])


def check_grads(grads, aux, nets, tag):
    """grads[net][name] against the oracle's aux[f"{net}_grads"][name]: every row within TOL["grad"], no ReLU flip allowed."""
    for net in nets:
        for nm, ref in aux[f"{net}_grads"].items():
            ok, overall, bad = grad_close(grads[net][nm], ref, TOL["grad"], max_flips=0)
            assert ok, (tag, net, nm, overall, bad)


def oracle_step(agent, st, case, b, hint=None, per_weights=None):
    """One oracle step on the masks the device used; every unit outside the rounding band must agree."""
    hint = hint or relu_hint(agent, case)
    ref, aux = O.update_parameters(st, b, per_weights=per_weights, return_aux=True, relu_hint=hint)
    assert hint.mismatch == 0, (hint.mismatch, hint.adopted, hint.ambiguous)
    return ref, aux


def check_state(agent, st):
    """All five nets, the Adam moments and step counts of the three optimizers, alpha -- after st.q1_opt.step steps.

    Adam moves every weight by ~lr per step whatever |g| is: weights are compared in units of lr (0.02 lr per step, at most a fraction
    5e-3 of the elements outside).  A Polyak target moves by only tau (w - w_t) per step, far inside that budget (a skipped or stale
    Polyak step would pass it), so the targets also get the budget scaled by tau (an error of the online weights reaches the target
    through tau), plus a few ulp of fp32 rounding per step."""
    steps = st.q1_opt.step
    budget = TOL["budget"] * st.lr * steps + 1e-7
    for net in NETS:
        mine = net_params(agent, net)
        for nm, ref in getattr(st, net).items():
            frac_bad = np.mean(np.abs(mine[nm] - ref) > budget)
            assert frac_bad < TOL["frac"], (net, nm, frac_bad, np.abs(mine[nm] - ref).max())
            if net.endswith("_target"):
                tb = st.tau * steps * budget + 4 * steps * np.spacing(np.abs(ref))
                frac_bad = np.mean(np.abs(mine[nm] - ref) > tb)
                assert frac_bad < TOL["frac"], ("polyak", net, nm, frac_bad, np.abs(mine[nm] - ref).max())
    for net, opt in (("policy", st.policy_opt), ("q1", st.q1_opt), ("q2", st.q2_opt)):
        sd = getattr(agent, f"{net}_optimizer").state_dict()
        for i, nm in enumerate(getattr(st, net)):
            assert int(sd["state"][i]["step"]) == opt.step, (net, nm, sd["state"][i]["step"], opt.step)
            assert grad_close(sd["state"][i]["exp_avg"].cpu().numpy(), opt.m[nm], TOL["adam"], max_flips=0)[0], (net, nm)
            assert grad_close(sd["state"][i]["exp_avg_sq"].cpu().numpy(), opt.v[nm], 2 * TOL["adam"], max_flips=0)[0], (net, nm)
    a = alpha_of(agent)
    assert abs(a - st.alpha) <= 1e-5 * abs(st.alpha), (a, st.alpha)


def n_stages_latency_form(hw, case, b, monkeypatch, **update_kw):
    """Stage count of the same program built under SACB_NO_STREAM (read whenever a program is built): the latency form."""
    with monkeypatch.context() as mp:
        mp.setenv("SACB_NO_STREAM", "1")
        agent, _ = make_agent(hw, case, math="bf16x3")
        agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), **update_kw)
        return agent.stats()["n_stages"]


# ---- A. fused-Adam update, throughput form ---------------------------------------------------------------------------------------
# 3000: ragged 128-row tiles, a ragged last K block of the dW GEMMs (3000 % 64 = 56) and ragged 16-row loss tiles.
# The critics' fc1 has obs + act = 365 inputs: its Adam epilogue runs the scalar pass B on every row.
THROUGHPUT = [("c2_humanoid_m2", 2048, 3, 81), ("c2_humanoid_m2", 3000, 3, 82), ("c2_humanoid_m2", 8192, 2, 83), ("c1_bipedal_m1", 4096, 3, 84)]


@pytest.mark.parametrize("name,B,steps,seed", THROUGHPUT)
def test_throughput_update_matches_oracle(hw, monkeypatch, name, B, steps, seed):
    """Every step against the oracle (losses, every gradient, alpha), then the whole state: all five nets, the Adam moments.
    Step 1 derives the shadows; from step 2 on the resident program reads what the Adam epilogues wrote."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    case = case_of(name, B, steps, seed)
    agent, st = make_agent(hw, case, math="bf16x3")
    for step in range(steps):
        b = batch_of(case, step)
        got = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=True)
        if step == 0:
            n_stages = agent.stats()["n_stages"]      # the handle holds this one program so far
        ref, aux = oracle_step(agent, st, case, b)
        check_losses(got, ref, step)
        check_grads({net: agent.exported_grads(net) for net in ("q1", "q2", "policy")}, aux, ("q1", "q2", "policy"), step)
        a = alpha_of(agent)
        assert abs(a - st.alpha) <= 1e-5 * abs(st.alpha), (step, a, st.alpha)
    check_state(agent, st)
    # the program really took the throughput form: it has more stages than the latency form (mixed stages are cut in two)
    b = batch_of(case, 0)
    assert n_stages > n_stages_latency_form(hw, case, b, monkeypatch, export_grads=True), n_stages


def _run(hw, case, steps, mode):
    agent, _ = make_agent(hw, case, math="bf16x3")
    losses = []
    for step in range(steps):
        b = batch_of(case, step)
        if mode == "rederive":
            agent.invalidate_shadows()
        losses.append(agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=(mode == "export")))
    out = {net: net_params(agent, net) for net in NETS}
    for net in ("policy", "q1", "q2"):
        sd = getattr(agent, f"{net}_optimizer").state_dict()["state"]
        out[f"{net}_opt"] = {f"{i}/{k}": sd[i][k].cpu().numpy() for i in sd for k in ("exp_avg", "exp_avg_sq")}
    return losses, alpha_of(agent), out


@pytest.mark.parametrize("B", [3000, 8192])
def test_throughput_update_bitwise_equalities(hw, monkeypatch, B):
    """Nothing on the fused-Adam path is order-dependent, so these runs must agree bit for bit over 4 steps:
    * a second identical handle (no atomics on this path);
    * the program that also exports gradients (it applies Adam as well, so it does not split K either);
    * invalidate_shadows() before every step, i.e. every shadow re-derived from the fp32 weights instead of read as the previous
      step's Adam epilogues left it (the throughput-form twin of test_resident_shadows_equal_rederived_shadows)."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    case = case_of("c2_humanoid_m2", B, 4, 85)
    l0, a0, s0 = _run(hw, case, 4, "plain")
    for mode in ("plain", "export", "rederive"):
        l1, a1, s1 = _run(hw, case, 4, mode)
        assert l1 == l0, (mode, l0, l1)
        assert a1 == a0, (mode, a0, a1)
        for grp in s0:
            for k in s0[grp]:
                np.testing.assert_array_equal(s1[grp][k], s0[grp][k], err_msg=f"{mode}: {grp} {k}")


def test_throughput_is_weighted_loss_and_td(hw, monkeypatch):
    """IS-weighted critic loss at B = 3000 with the TD errors read back: the loss task's 16-row tiles end in a ragged tail."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    case = case_of("c2_humanoid_m2", 3000, 2, 86)
    agent, st = make_agent(hw, case, math="bf16x3")
    rng = np.random.RandomState(7)
    for step in range(case["steps"]):
        b = batch_of(case, step)
        w = rng.uniform(0.2, 1.0, case["batch"]).astype(np.float32)
        got, td = agent.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), is_weights=w, want_td=True, export_grads=True)
        ref, aux = oracle_step(agent, st, case, b, per_weights=w)
        check_losses(got, ref, step)
        check_grads({net: agent.exported_grads(net) for net in ("q1", "q2", "policy")}, aux, ("q1", "q2", "policy"), step)
        want = np.abs(aux["td1"])
        assert td.shape == want.shape
        # |q1 - y| per row: within the loss tolerance of the scale of y (q1 and y each carry that relative error)
        np.testing.assert_allclose(td, want, rtol=TOL["loss"], atol=TOL["loss"] * float(np.sqrt(np.mean(aux["y"] ** 2))), err_msg=f"step {step}")
    check_state(agent, st)


# ---- B. data-parallel backward, world = 1 -----------------------------------------------------------------------------------------
def _dp_agent(hw, case, b, capacity=None):
    agent, st = make_agent(hw, case, math="bf16x3", capacity=capacity or case["batch"])
    agent.replay_buffer.push_many(b["s"], b["a"], b["r"], b["s2"], b["d"])
    return hw.distributed.DataParallelSAC(agent), st


def _dp_backward(hw, dp, phase, rows, b, no_stream=False):
    """sacb_dp_backward on ring positions `rows` (the batch was pushed in order); the program is built on the first call of a phase,
    under SACB_NO_STREAM when no_stream."""
    N = hw._native
    e = (N.f32(b["eps_next"][rows]), N.f32(b["eps_cur"][rows]))
    with pytest.MonkeyPatch.context() as mp:
        if no_stream:
            mp.setenv("SACB_NO_STREAM", "1")
        else:
            mp.delenv("SACB_NO_STREAM", raising=False)
        N.check(N.lib().sacb_dp_backward(dp.agent._h, phase, rows.size, N.ptr(rows, ctypes.c_int64) if phase == 0 else None, N.ptr(e[0]), N.ptr(e[1])))
    dp.agent.synchronize()


def _dp_apply(hw, dp, phase):
    torch.cuda.synchronize()      # torch-side writes of the slabs (default stream) before the library's stream reads them
    hw._native.check(hw._native.lib().sacb_dp_apply(dp.agent._h, phase))
    dp.agent.synchronize()


def _phase_grads(dp, phase):
    nets = ("q1", "q2") if phase == 0 else ("policy",)
    g = {net: dp.agent.exported_grads(net) for net in nets}
    if phase == 1:
        g["log_alpha"] = float(dp.gradient_slabs(1)[1][0].item())
    return g


def _local_losses(hw, dp):
    losses = np.zeros(3, np.float32)
    hw._native.check(hw._native.lib().sacb_get_losses(dp.agent._h, 0, hw._native.ptr(losses)))
    return dict(zip(("q1_loss", "q2_loss", "policy_loss"), losses.tolist()))


def _close_split(a, b, tag):
    for net in a:
        if net == "log_alpha":
            assert abs(a[net] - b[net]) <= SPLIT_TOL * abs(b[net]) + 1e-9, (tag, a[net], b[net])
            continue
        for nm in a[net]:
            e = relerr(a[net][nm], b[net][nm])
            assert e < SPLIT_TOL, (tag, net, nm, e)


def _close_oracle(grads, aux, nets, tag):
    for net in nets:
        for nm, ref in aux[f"{net}_grads"].items():
            e = relerr(grads[net][nm], ref)
            assert e < SPLIT_ORACLE_TOL, (tag, net, nm, e)


def _check_log_alpha_grad(g, aux):
    # -mean(logp + target_entropy): logp carries the loss tolerance per row, so the bound scales with mean |logp|
    ref = float(aux["log_alpha_grad"][0])
    assert abs(g - ref) <= TOL["grad"] * (abs(ref) + float(np.mean(np.abs(aux["logp"])))), (g, ref)


def _merged_hint(masks_phase0, agent, case):
    # the critic masks on (s, a) are read after phase 0; the policy and the post-step critics on (s, a_new) after phase 1
    hint = relu_hint(agent, case)
    hint.masks.update({k: v for k, v in masks_phase0.items() if k[0] in ("q1", "q2")})
    return hint


# local batch -> dW K chunks (B / 64 K blocks, at least 16 blocks and at most 16 chunks) and 1024-row column-sum chunks:
#   2048 -> 2 / 2, 3000 -> 2 (the second ragged: 23 blocks, the last of 56 rows) / 3, 8192 -> 8 / 8, 65536 -> 16 / 64
@pytest.mark.parametrize("B", [2048, 3000, 8192, 65536])
def test_dp_backward_matches_oracle_and_unsplit_program(hw, B):
    """One data-parallel step on one replica, every phase by hand through the ABI (backward -> slab -> apply):
    * each backward twice: the slab is zeroed first, so the second equals the first (not twice it);
    * against the same program built under SACB_NO_STREAM (latency form: no split K; the same forward bit for bit): the losses, and
      up to B = UNSPLIT_MAX_K every gradient tensor to 2e-5;
    * against the oracle: every gradient tensor to 4e-5 (SPLIT_ORACLE_TOL) besides the row-wise 3e-4, log_alpha's gradient, the
      losses, and after both applies the whole state."""
    case = case_of("c2_humanoid_m2", B, 1, 87)
    b = batch_of(case, 0)
    rows = np.arange(B, dtype=np.int64)
    dp, st = _dp_agent(hw, case, b)
    lat, _ = _dp_agent(hw, case, b)
    grads = {}
    for phase in (0, 1):
        _dp_backward(hw, dp, phase, rows, b)
        first = _phase_grads(dp, phase)
        _dp_backward(hw, dp, phase, rows, b)
        grads[phase] = _phase_grads(dp, phase)
        _close_split(grads[phase], first, f"phase {phase} twice")
        if phase == 0:
            masks0 = relu_hint(dp.agent, case).masks
        _dp_backward(hw, lat, phase, rows, b, no_stream=True)
        if B <= UNSPLIT_MAX_K:
            _close_split(grads[phase], _phase_grads(lat, phase), f"phase {phase} vs unsplit")
        for mine, other in zip(dp.gradient_slabs(phase), lat.gradient_slabs(phase)):      # both replicas step on the same gradients
            other.copy_(mine)
        _dp_apply(hw, dp, phase)
        _dp_apply(hw, lat, phase)
    assert dp.agent.stats()["n_stages"] > lat.agent.stats()["n_stages"]      # the split program really is the throughput form
    got = _local_losses(hw, dp)
    for k, v in _local_losses(hw, lat).items():
        assert abs(got[k] - v) <= SPLIT_TOL * abs(v) + 1e-7, (k, got[k], v)
    hint = _merged_hint(masks0, dp.agent, case)
    ref, aux = oracle_step(dp.agent, st, case, b, hint=hint)
    check_losses(got, ref, "dp")
    check_grads(grads[0], aux, ("q1", "q2"), "phase 0")
    check_grads(grads[1], aux, ("policy",), "phase 1")
    _close_oracle(grads[0], aux, ("q1", "q2"), "phase 0")
    _close_oracle(grads[1], aux, ("policy",), "phase 1")
    _check_log_alpha_grad(grads[1]["log_alpha"], aux)
    check_state(dp.agent, st)


def test_dp_two_shards_equal_fused_update(hw):
    """Two replicas of B_local = 4096 (8 K chunks, 4 column-sum chunks each), slabs averaged by hand as the all-reduce would: against
    the fused update on the concatenated 8192 rows and against the oracle."""
    B, half = 8192, 4096
    case = case_of("c2_humanoid_m2", B, 1, 88)
    b = batch_of(case, 0)
    full, st = make_agent(hw, case, math="bf16x3")
    got_full = full.update_from_batch(b, eps=(b["eps_next"], b["eps_cur"]), export_grads=True)
    ref, aux = oracle_step(full, st, case, b)
    check_losses(got_full, ref, "fused")
    shards = [_dp_agent(hw, dict(case, batch=half), b, capacity=B)[0] for _ in range(2)]
    rows = [np.arange(0, half, dtype=np.int64), np.arange(half, B, dtype=np.int64)]
    grads = {}
    for phase in (0, 1):
        for r, dp in enumerate(shards):
            _dp_backward(hw, dp, phase, rows[r], b)
        torch.cuda.synchronize()
        for s0, s1 in zip(shards[0].gradient_slabs(phase), shards[1].gradient_slabs(phase)):
            m = (s0 + s1) / 2
            s0.copy_(m); s1.copy_(m)
        torch.cuda.synchronize()
        grads[phase] = _phase_grads(shards[0], phase)
        for dp in shards:
            _dp_apply(hw, dp, phase)
    check_grads(grads[0], aux, ("q1", "q2"), "phase 0")
    check_grads(grads[1], aux, ("policy",), "phase 1")
    _close_oracle(grads[0], aux, ("q1", "q2"), "phase 0")
    _close_oracle(grads[1], aux, ("policy",), "phase 1")
    _check_log_alpha_grad(grads[1]["log_alpha"], aux)
    l0, l1 = _local_losses(hw, shards[0]), _local_losses(hw, shards[1])
    check_losses({k: (l0[k] + l1[k]) / 2 for k in l0}, ref, "two shards")
    lr = st.lr
    for net in NETS:
        want = net_params(full, net)
        for r, dp in enumerate(shards):
            mine = net_params(dp.agent, net)
            for nm in want:
                # Adam's first step is sign-like: a gradient within rounding of zero may step by +lr in one run and -lr in the other
                assert np.mean(np.abs(mine[nm] - want[nm]) > 0.02 * lr) < 5e-3, (net, nm, r)
    for net in NETS:
        p0, p1 = net_params(shards[0].agent, net), net_params(shards[1].agent, net)
        for nm in p0:
            np.testing.assert_array_equal(p0[nm], p1[nm], err_msg=f"replicas diverged: {net}.{nm}")
    check_state(shards[0].agent, st)
