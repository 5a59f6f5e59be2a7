"""Shared helpers of the GPU parity tests: load an oracle state into the product SAC, compare tensors."""
import numpy as np
import torch

from oracle import sac_oracle_np as O

# Relative tolerances of the parity tests.  Both math modes read the same bf16 hi/lo pair operands; the budget is in units of lr per step.
PARITY_TOL = {"fp32": dict(loss=3e-4, grad=3e-4, adam=6e-4, frac=5e-3, budget=0.02),
              "bf16x3": dict(loss=3e-4, grad=3e-4, adam=6e-4, frac=5e-3, budget=0.02)}
TOL = PARITY_TOL["bf16x3"]
NETS = ("policy", "q1", "q2", "q1_target", "q2_target")


def relerr(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def make_agent(hw, case, math="fp32", launch="staged", **kw):
    """Product SAC holding exactly the numpy-seeded weights of oracle make_state(case)."""
    hw.use_networks("model1" if case["n_hidden"] == 2 else "model2")
    st = O.make_state(case["obs"], case["act"], case["hidden"], case["n_hidden"], seed=case["seed"],
                      bias_scale=case.get("bias_scale", 0.0), head_scale=case.get("head_scale", 1.0),
                      automatic_entropy_tuning=case.get("auto_entropy", True))
    agent = hw.SAC(case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", math=math, launch=launch,
                   automatic_entropy_tuning=case.get("auto_entropy", True), max_batch=max(case["batch"], 16),
                   capacity=kw.pop("capacity", 4096), seed=1234, **kw)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        getattr(agent, net).load_state_dict({k: torch.from_numpy(v.copy()) for k, v in getattr(st, net).items()})
    return agent, st


def relu_hint(agent, case, band=1e-4, band_post_adam=1e-2, agent_index=0):
    """ReLU masks the device used in the last update (tests/oracle ReluHint): the three differentiated passes.  `agent` is anything
    that holds a library handle `_h` (a SAC, a PopulationSAC); `agent_index` picks the member of a population.

    band: |z| < 1e-4 rms(z) may take either sign (bf16-pair operand storage, 2^-16 per element).  The actor phase
    evaluates the critics right AFTER their Adam step (sac_imp.py:109,113 -> :117-118): a weight whose gradient is
    within rounding of zero moves by +lr or -lr (early Adam steps are sign-like), shifting a pre-activation by up to
    2*lr*|x|; those two passes get the wider band."""
    import ctypes
    from humanoid_walking_with_sac_b200 import _native as N
    B, H, nh = case["batch"], case["hidden"], case["n_hidden"]
    masks = {}
    buf = np.empty((B, H), np.float32)
    for layer in range(nh):
        for tag, group, k in (("policy", 0, 0), ("q1", 1, 0), ("q2", 1, 1), ("q1a", 2, 0), ("q2a", 2, 1)):
            N.check(N.lib().sacb_debug_read_activation(agent._h, agent_index, group, k, layer, B, N.ptr(buf)))
            masks[(tag, layer + 1)] = buf > 0
    return O.ReluHint(masks, band, {"q1a": band_post_adam, "q2a": band_post_adam})


def oracle_step(agent, st, case, b, hint=None, per_weights=None):
    """One oracle step on the masks the device used; every unit outside the rounding band must agree."""
    hint = hint or relu_hint(agent, case)
    ref, aux = O.update_parameters(st, b, per_weights=per_weights, return_aux=True, relu_hint=hint)
    assert hint.mismatch == 0, (hint.mismatch, hint.adopted, hint.ambiguous)
    return ref, aux


def check_losses(got, ref, tag):
    for k in ("q1_loss", "q2_loss", "policy_loss"):
        assert abs(got[k] - ref[k]) <= TOL["loss"] * abs(ref[k]) + 1e-6, (tag, k, got[k], ref[k])


def alpha_of(agent):
    a = agent.alpha
    return float(a) if not hasattr(a, "item") else float(a.item())


def sac_state(agent):
    """Learner state of a SAC in the layout check_state reads: {net: {name: array}}, {opt: (step, m, v)} for the three optimizers
    (keyed f"{net}_opt", m / v by parameter name), "alpha"."""
    out = {net: net_params(agent, net) for net in NETS}
    for net in ("policy", "q1", "q2"):
        sd = getattr(agent, f"{net}_optimizer").state_dict()["state"]
        names = list(out[net])
        steps = {int(sd[i]["step"]) for i in sd}
        assert len(steps) == 1, (net, steps)      # one step count per optimizer
        out[f"{net}_opt"] = (steps.pop(), {nm: sd[i]["exp_avg"].cpu().numpy() for i, nm in enumerate(names)},
                             {nm: sd[i]["exp_avg_sq"].cpu().numpy() for i, nm in enumerate(names)})
    out["alpha"] = alpha_of(agent)
    return out


def population_state(pop, agent):
    """The same layout for member `agent` of a PopulationSAC, read through the C ABI (sacb_export_tensor / sacb_get_scalars)."""
    import ctypes
    from humanoid_walking_with_sac_b200 import _native as N
    lib = N.lib()

    def export(net_id, slot):
        d = {}
        for t, (nm, shape) in enumerate(pop._names[net_id]):
            host = np.empty(shape, np.float32)
            N.check(lib.sacb_export_tensor(pop._h, int(agent), net_id, slot, t, N.ptr(host), host.size))
            d[nm] = host
        return d
    sc = N.Scalars()
    N.check(lib.sacb_get_scalars(pop._h, int(agent), ctypes.byref(sc)))
    out = {net: export(net_id, N.SLOT_PARAM) for net_id, net in enumerate(NETS)}
    for net_id, net, step in ((N.NET_POLICY, "policy", sc.step_policy), (N.NET_Q1, "q1", sc.step_q1), (N.NET_Q2, "q2", sc.step_q2)):
        out[f"{net}_opt"] = (int(step), export(net_id, N.SLOT_ADAM_M), export(net_id, N.SLOT_ADAM_V))
    out["alpha"] = float(sc.alpha)
    return out


def arena_offset(pop, agent):
    """Bytes from agent 0's arena to `agent`'s (the device address of its first policy weight)."""
    import ctypes
    from humanoid_walking_with_sac_b200 import _native as N
    p0, p = ctypes.c_void_p(), ctypes.c_void_p()
    N.check(N.lib().sacb_tensor_dev(pop._h, 0, N.NET_POLICY, N.SLOT_PARAM, 0, ctypes.byref(p0)))
    N.check(N.lib().sacb_tensor_dev(pop._h, int(agent), N.NET_POLICY, N.SLOT_PARAM, 0, ctypes.byref(p)))
    return p.value - p0.value


def selected_agents(pop, require_far=False):
    """0, 1, the last agent, and the first agents whose arena starts more than 2^31 / 2^32 bytes past agent 0's."""
    n = len(pop)
    offs = [arena_offset(pop, i) for i in range(n)]
    far = [next((i for i in range(n) if offs[i] > lim), None) for lim in (1 << 31, 1 << 32)]
    if require_far:
        assert None not in far, (offs[-1], far)
    return sorted({0, 1, n - 1, *(i for i in far if i is not None)})


def check_state(got, st):
    """All five nets, the Adam moments and step counts of the three optimizers, alpha -- after st.q1_opt.step steps.  `got` is a
    snapshot in the layout of sac_state / population_state.

    Adam moves every weight by ~lr per step whatever |g| is: weights are compared in units of lr (0.02 lr per step, at most a fraction
    5e-3 of the elements outside).  A Polyak target moves by only tau (w - w_t) per step, far inside that budget (a skipped or stale
    Polyak step would pass it), so the targets also get the budget scaled by tau (an error of the online weights reaches the target
    through tau), plus a few ulp of fp32 rounding per step."""
    steps = st.q1_opt.step
    budget = TOL["budget"] * st.lr * steps + 1e-7
    for net in NETS:
        mine = got[net]
        for nm, ref in getattr(st, net).items():
            frac_bad = np.mean(np.abs(mine[nm] - ref) > budget)
            assert frac_bad < TOL["frac"], (net, nm, frac_bad, np.abs(mine[nm] - ref).max())
            if net.endswith("_target"):
                tb = st.tau * steps * budget + 4 * steps * np.spacing(np.abs(ref))
                frac_bad = np.mean(np.abs(mine[nm] - ref) > tb)
                assert frac_bad < TOL["frac"], ("polyak", net, nm, frac_bad, np.abs(mine[nm] - ref).max())
    for net, opt in (("policy", st.policy_opt), ("q1", st.q1_opt), ("q2", st.q2_opt)):
        step, m, v = got[f"{net}_opt"]
        assert step == opt.step, (net, step, opt.step)
        for nm in getattr(st, net):
            assert grad_close(m[nm], opt.m[nm], TOL["adam"], max_flips=0)[0], (net, nm)
            assert grad_close(v[nm], opt.v[nm], 2 * TOL["adam"], max_flips=0)[0], (net, nm)
    assert abs(got["alpha"] - st.alpha) <= 1e-5 * abs(st.alpha), (got["alpha"], st.alpha)


def batch_of(case, step):
    return O.make_batch(case["obs"], case["act"], case["batch"], seed=case["seed"] * 100 + step)


def net_params(agent, net):
    return {k: v.detach().cpu().numpy() for k, v in getattr(agent, net).state_dict().items()}


def grad_close(got, ref, tol, max_flips=2):
    """Gradient parity that tolerates a couple of ReLU mask flips.

    A hidden unit whose pre-activation lies within rounding (~1e-6) of zero for one sample is on for one
    summation order and off for another; the reference itself flips such units when its BLAS changes.  One flip
    moves one row of that layer's weight gradient (and one bias entry) by O(1/B).  So: every row of the tensor must
    match within `tol` (relative to the RMS row norm) except at most `max_flips` rows, and the whole tensor within 5e-2."""
    got = np.asarray(got, np.float64).reshape(np.asarray(ref).shape)
    ref = np.asarray(ref, np.float64)
    g2, r2 = (got.reshape(got.shape[0], -1), ref.reshape(ref.shape[0], -1)) if ref.ndim == 2 and ref.shape[0] > 1 else (got.reshape(-1, 1), ref.reshape(-1, 1))
    row_err = np.linalg.norm(g2 - r2, axis=1)
    scale = max(np.sqrt(np.mean(np.sum(r2 * r2, axis=1))), 1e-30)
    bad = int(np.sum(row_err > tol * scale * max(1.0, np.sqrt(r2.shape[0]) / 4)))
    overall = relerr(got, ref)
    ok = overall < tol or (bad <= max_flips and overall < 5e-2)
    return ok, overall, bad


def state_from_checkpoint(path, case, alpha_from_file=True):
    """Oracle SACState holding the networks of a reference-format `save()` / `save_checkpoint()` file (sac_imp.py:154-233)."""
    ck = torch.load(path, map_location="cpu", weights_only=False)
    st = O.make_state(case["obs"], case["act"], case["hidden"], case["n_hidden"], seed=0)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        setattr(st, net, {k: v.detach().cpu().numpy().astype(np.float32).copy() for k, v in ck[f"{net}_state_dict"].items()})
    if alpha_from_file:
        a = ck["alpha"]
        st.alpha = float(a.detach().reshape(-1)[0]) if torch.is_tensor(a) else float(a)
    for net, opt in (("policy", "policy_opt"), ("q1", "q1_opt"), ("q2", "q2_opt")):
        sd = ck.get(f"{net}_optimizer_state_dict")
        if sd and sd["state"]:
            names = list(getattr(st, net).keys())
            o = getattr(st, opt)
            for i, nm in enumerate(names):
                o.m[nm] = sd["state"][i]["exp_avg"].cpu().numpy().copy()
                o.v[nm] = sd["state"][i]["exp_avg_sq"].cpu().numpy().copy()
            o.step = int(float(sd["state"][0]["step"]))
    if "log_alpha" in ck:
        st.log_alpha = ck["log_alpha"].detach().cpu().numpy().astype(np.float32).reshape(1).copy()
        sd = ck.get("alpha_optimizer_state_dict")
        if sd and sd["state"]:
            st.alpha_opt.m["log_alpha"] = sd["state"][0]["exp_avg"].cpu().numpy().reshape(1).copy()
            st.alpha_opt.v["log_alpha"] = sd["state"][0]["exp_avg_sq"].cpu().numpy().reshape(1).copy()
            st.alpha_opt.step = int(float(sd["state"][0]["step"]))
    return st, ck
