"""Per-agent prioritized replay in a population (PopulationSAC(replay="per")): one sampler chain and one priority write-back for all
agents.  Every agent's sample is bit-exact against the C oracle and equal to a one-agent handle's; the learner step equals independent
single-agent SAC learners bit for bit.  Reference: replay_buffer.py:25-90 per agent, sac_imp.py:74-144 per agent."""
import ctypes

import numpy as np
import pytest

from oracle import per_oracle as PO
from tests.golden import cases
from tests.test_oracle_per_golden import ulp_diff
from tests.util import check_losses, check_state, make_agent, oracle_step, population_state, relu_hint, sac_state

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
DEFAULT_SEED = 0x5AC0B200      # sacb_default_config's seed: what a standalone PrioritizedReplayBuffer draws with


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    hw.use_networks("model1")
    yield hw
    hw.use_networks("model1")


# ---- numpy restatement of the device-drawn uniforms (include/sacb200.h, sacb_per_sample) ------------------------------------------------
def _mix(x):
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & M64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def agent_key(seed, a):
    """seed for agent 0, seed ^ splitmix64(a) otherwise."""
    return seed if a == 0 else seed ^ _mix((a + 0x9E3779B97F4A7C15) & M64)


def device_uniforms(key, frame, k):
    return np.array([(_mix(key ^ ((frame * 0x9E3779B97F4A7C15 + j * 0xBF58476D1CE4E5B9) & M64)) >> 11) * (1.0 / 9007199254740992.0)
                     for j in range(k)], np.float64)


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def per_pop(hw, n, capacity, B, obs=3, act=2, seed=DEFAULT_SEED, **kw):
    return hw.PopulationSAC(n, obs, act, hidden_dim=16, device="cuda", capacity=capacity, max_batch=B, replay="per", seed=seed, **kw)


def push_zero_rows(hw, h, agent, n):
    """n zero transitions into one agent's ring (only the priority tables matter to the sampler tests)."""
    N = hw._native
    lib = N.lib()
    rows = np.zeros((n, int(lib.sacb_row_floats(h))), np.float32)
    N.check(lib.sacb_push_rows(h, agent, N.ptr(rows), n))


def single_buffer(hw, capacity, n_pushed):
    """A standalone PrioritizedReplayBuffer with the same ring state as a population agent that got n_pushed zero rows."""
    buf = hw.PrioritizedReplayBuffer(capacity)
    buf.push_many(np.zeros((1, 3)), np.zeros((1, 2)), np.zeros(1), np.zeros((1, 3)), np.zeros(1))
    push_zero_rows(hw, buf._h, 0, n_pushed - 1)
    return buf


def tables(lengths, dists, seed0):
    out = []
    for a, (m, dist) in enumerate(zip(lengths, dists)):
        pri = cases.per_priorities(dict(n=m, capacity=m, seed=seed0 + a, dist=dist))
        out.append((pri, (pri ** np.float32(0.6)).astype(np.float32)))
    return out


def sample_all(hw, pop, B, u=None):
    N = hw._native
    idx, w = np.empty((pop.n_agents, B), np.int64), np.empty((pop.n_agents, B), np.float32)
    uu = None if u is None else np.ascontiguousarray(u, np.float64)
    N.check(N.lib().sacb_per_sample_all(pop._h, N.ptr(uu, ctypes.c_double), B, N.ptr(idx, ctypes.c_int64), N.ptr(w)))
    return idx, w


def stats(hw, h, agent):
    N = hw._native
    st = N.PerStats()
    N.check(N.lib().sacb_per_get_stats(h, agent, ctypes.byref(st)))
    return st


def read_slots(hw, h, agent, B):
    N = hw._native
    out = np.empty(B, np.int32)
    N.check(N.lib().sacb_debug_read_slots(h, agent, N.ptr(out, ctypes.c_int32), B))
    return out


CAP, B5 = 50000, 256
# agent 0 wrapped (pushed past capacity), 1 partly filled, 2 holds exactly B, 3 full, 4 partly filled
PUSHED = [CAP + 3000, 30001, B5, CAP, 12345]
DISTS = ["halfnormal", "floor1pct", "lognormal3", "fresh", "halfnormal"]


def five_agents(hw):
    pop = per_pop(hw, 5, CAP, B5)
    lens = [min(p, CAP) for p in PUSHED]
    for a, p in enumerate(PUSHED):
        push_zero_rows(hw, pop._h, a, p)
        assert pop.buffer_len(a) == lens[a]
    tabs = tables(lens, DISTS, 70)
    for a, (pri, pa) in enumerate(tabs):
        pop.set_priorities(a, pri, pa)
    return pop, tabs


# ---- 1. sampler against the C oracle --------------------------------------------------------------------------------------------------
def test_population_sampler_matches_oracle(hw):
    pop, tabs = five_agents(hw)
    frame0 = [1 + 1000 * a for a in range(5)]      # every agent its own beta
    for a in range(5):
        pop.set_frame(a, frame0[a])
    rng = np.random.RandomState(3)
    for call in range(3):
        u = rng.random_sample((5, B5))
        idx, w = sample_all(hw, pop, B5, u)
        for a, (_, pa) in enumerate(tabs):
            ref_idx, ref_w = PO.sample(pa, u[a], PO.beta(frame0[a] + call))
            np.testing.assert_array_equal(idx[a], ref_idx, err_msg=f"call {call} agent {a}")
            assert ulp_diff(w[a], ref_w).max() <= 16, (call, a)
            np.testing.assert_array_equal(read_slots(hw, pop._h, a, B5), ref_idx.astype(np.int32))
    for a, (_, pa) in enumerate(tabs):
        st = stats(hw, pop._h, a)
        assert st.total_f32 == pa.sum(), a
        assert st.frame == frame0[a] + 3 == pop.frame(a)


# ---- 2. the exact pass runs for the agent that needs it only ------------------------------------------------------------------------------
def test_exact_pass_in_one_agent_only(hw):
    n, B = 50000, 256
    pop = per_pop(hw, 3, n, B)
    tabs = tables([n] * 3, ["lognormal3"] * 3, 39)      # agent 2: the set of test_per_ambiguous_samples_take_the_exact_path (fine elements)
    for a, (pri, pa) in enumerate(tabs):
        push_zero_rows(hw, pop._h, a, n)
        pop.set_priorities(a, pri, pa)
    rng = np.random.RandomState(8)
    u = rng.random_sample((3, B))
    _, _, _, cdf = PO.sample(tabs[2][1], np.array([0.5]), 0.4, want_tables=True)
    u2 = cdf[np.random.RandomState(1).randint(0, n - 1, B)].copy()      # agent 2: u ON cdf boundaries
    u2[::2] = np.nextafter(u2[::2], 0.0)
    u[2] = u2
    before = [stats(hw, pop._h, a).n_exact_fallbacks for a in range(3)]
    idx, _ = sample_all(hw, pop, B, u)
    after = [stats(hw, pop._h, a) for a in range(3)]
    for a, (_, pa) in enumerate(tabs):
        np.testing.assert_array_equal(idx[a], PO.sample(pa, u[a], PO.beta(1))[0], err_msg=f"agent {a}")
    assert after[2].n_fine > 0 and after[2].n_flagged > 0 and after[2].n_exact_fallbacks >= before[2] + 1
    assert [after[a].n_exact_fallbacks for a in (0, 1)] == [before[0], before[1]]


# ---- 3. population sample == one-agent handles ----------------------------------------------------------------------------------------------
def test_population_sample_equals_single_handles(hw):
    pop, tabs = five_agents(hw)
    singles = []
    for a, p in enumerate(PUSHED):
        buf = single_buffer(hw, CAP, p)
        buf.set_priorities(*tabs[a])
        singles.append(buf)
    rng = np.random.RandomState(4)
    for call in range(2):
        u = rng.random_sample((5, B5))
        idx, w = sample_all(hw, pop, B5, u)
        for a, buf in enumerate(singles):
            *_, ref_idx, ref_w = buf.sample(B5, u=u[a])
            np.testing.assert_array_equal(idx[a], ref_idx, err_msg=f"call {call} agent {a}")
            np.testing.assert_array_equal(w[a], ref_w, err_msg=f"call {call} agent {a}")
    # one agent of the population sampled alone is the chain over that agent
    u = rng.random_sample(B5)
    *_, i3, w3 = pop.sample(3, B5, u=u)
    *_, r3, rw3 = singles[3].sample(B5, u=u)
    np.testing.assert_array_equal(i3, r3)
    np.testing.assert_array_equal(w3, rw3)


# ---- 4. device-drawn uniforms: per-agent keys -----------------------------------------------------------------------------------------------
def test_device_uniforms_follow_the_documented_keys(hw):
    pop, tabs = five_agents(hw)
    single = single_buffer(hw, CAP, PUSHED[0])
    single.set_priorities(*tabs[0])
    N = hw._native
    for call in range(2):
        idx, _ = sample_all(hw, pop, B5)
        ref0 = np.empty(B5, np.int64)
        N.check(N.lib().sacb_per_sample(single._h, 0, None, B5, N.ptr(ref0, ctypes.c_int64), None, None, None, None, None, None))
        np.testing.assert_array_equal(idx[0], ref0, err_msg=f"call {call}")      # agent 0 draws what a one-agent handle draws
        for a, (_, pa) in enumerate(tabs):
            u = device_uniforms(agent_key(DEFAULT_SEED, a), 1 + call, B5)
            np.testing.assert_array_equal(idx[a], PO.sample(pa, u, PO.beta(1 + call))[0], err_msg=f"call {call} agent {a}")
    assert len({tuple(r[:16]) for r in idx}) == 5      # distinct streams


# ---- 5. push and write-back rules per agent ----------------------------------------------------------------------------------------------
def test_push_and_update_rules_per_agent(hw):
    cap, n = 64, 3
    pop = per_pop(hw, n, cap, 16)
    ref = [np.zeros(cap, np.float32) for _ in range(n)]
    length, pos = [0] * n, [0] * n

    def push(a, k):
        rng = np.random.RandomState(a * 100 + k)
        pop.push_many(a, rng.standard_normal((k, 3)), rng.standard_normal((k, 2)), np.zeros(k), rng.standard_normal((k, 3)), np.zeros(k))
        for _ in range(k):
            pos[a] = PO.push(ref[a], length[a], pos[a])
            length[a] = min(cap, length[a] + 1)

    push(0, 10)
    push(1, 70)      # wraps
    for a, (idx, td) in enumerate(((np.array([1, 3, 3, 7, 1], np.int64), np.array([5.5, 0.25, 9.0, 2.0, 0.5], np.float32)),
                                   (np.array([0, 63, 12, 12], np.int64), np.array([0.125, 3.0, 0.75, 1.5], np.float32)))):
        pop.update_priorities(a, idx, td)      # duplicates: the last one wins
        PO.update_priorities(ref[a], idx, td)
    for a in range(n):
        np.testing.assert_array_equal(pop.priorities(a), ref[a], err_msg=f"agent {a} after update")
    assert ref[0].max() != ref[1].max()
    for a in range(n):
        push(a, 3)      # agents 0 and 1 write their own maximum, the empty agent 2 writes 1.0
        np.testing.assert_array_equal(pop.priorities(a), ref[a], err_msg=f"agent {a} after push")
    assert ref[2][0] == 1.0
    # float64 priorities: + 1e-6 in float64, then the float32 store
    pop.update_priorities(2, [0, 2, 0], np.array([0.3, 0.7, 0.9]))
    r = ref[2].copy()
    r[[2, 0]] = (np.array([0.7, 0.9]) + 1e-6).astype(np.float32)
    np.testing.assert_array_equal(pop.priorities(2), r)
    np.testing.assert_array_equal(pop.priorities(1), ref[1])
    # clearing one agent's replay clears its table only
    N = hw._native
    N.check(N.lib().sacb_clear_replay(pop._h, 1))
    np.testing.assert_array_equal(pop.priorities(1), np.zeros(cap, np.float32))
    np.testing.assert_array_equal(pop.priorities(0), ref[0])


# ---- 6. learner step == independent single-agent learners, bit for bit -------------------------------------------------------------------------
def import_nets(hw, pop, a, agent):
    N = hw._native
    lib = N.lib()
    for net_id, net in enumerate(("policy", "q1", "q2", "q1_target", "q2_target")):
        for t, (_, p) in enumerate(getattr(agent, net).named_parameters()):
            host = N.f32(p.detach().cpu().numpy())
            N.check(lib.sacb_import_tensor(pop._h, a, net_id, N.SLOT_PARAM, t, N.ptr(host), host.size))


def assert_same_learner(pop, a, single, tag):
    got, ref = population_state(pop, a), sac_state(single)
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        for nm, v in ref[net].items():
            np.testing.assert_array_equal(got[net][nm], v, err_msg=f"{tag} agent {a} {net}.{nm}")
    for opt in ("policy_opt", "q1_opt", "q2_opt"):
        assert got[opt][0] == ref[opt][0], (tag, a, opt)
        for k in (1, 2):
            for nm, v in ref[opt][k].items():
                np.testing.assert_array_equal(got[opt][k][nm], v, err_msg=f"{tag} agent {a} {opt}[{k}].{nm}")
    assert np.float32(got["alpha"]) == np.float32(ref["alpha"]), (tag, a)
    np.testing.assert_array_equal(pop.priorities(a), single.replay_buffer.priorities, err_msg=f"{tag} agent {a} priorities")


def test_learner_step_equals_single_agents(hw):
    case = cases.UPDATE_CASES["tiny_m2"]
    B, n, rows = case["batch"], 3, 40
    singles = [make_agent(hw, dict(case, seed=case["seed"] + 10 * a), math="bf16x3", capacity=64, replay="per", per_weighted_loss=True)[0]
               for a in range(n)]
    try:
        pop = hw.PopulationSAC(n, case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", capacity=64, max_batch=singles[0]._cfg.max_batch,
                               math="bf16x3", seed=1234, replay="per", per_weighted_loss=True)
        tabs = tables([rows] * n, ["halfnormal", "lognormal3", "floor1pct"], 90)
        for a, agent in enumerate(singles):
            import_nets(hw, pop, a, agent)
            d = cases.per_transitions(dict(n=rows, obs=case["obs"], act=case["act"], seed=80 + a))
            agent.replay_buffer.push_many(d["s"], d["a"], d["r"], d["s2"], d["d"])
            pop.push_many(a, d["s"], d["a"], d["r"], d["s2"], d["d"])
            agent.replay_buffer.set_priorities(*tabs[a])
            pop.set_priorities(a, *tabs[a])
        rng = np.random.RandomState(21)
        for step in range(3):
            u = rng.random_sample((n, B))
            e_next = rng.standard_normal((n, B, case["act"])).astype(np.float32)
            e_cur = rng.standard_normal((n, B, case["act"])).astype(np.float32)
            got = pop.update_parameters(B, u=u, eps=(e_next, e_cur))
            for a, agent in enumerate(singles):
                ref = agent.update_parameters(B, u=u[a], eps=(e_next[a], e_cur[a]))
                for k in ("q1_loss", "q2_loss", "policy_loss"):
                    assert np.float32(got[a][k]) == np.float32(ref[k]), (step, a, k, got[a][k], ref[k])
                assert_same_learner(pop, a, agent, f"step {step}")
                assert pop.frame(a) == agent.replay_buffer.frame == 2 + step
    finally:
        hw.use_networks("model1")


# ---- 7. C2 shape, device-drawn uniforms ----------------------------------------------------------------------------------------------------
def test_c2_population_step_with_device_draws(hw):
    case = cases.UPDATE_CASES["c2_humanoid_m2"]
    B, n, rows, cap, seed = case["batch"], 8, 600, 1024, 77
    N = hw._native
    lib = N.lib()
    keep = (0, 1, 7)
    try:
        singles = {a: make_agent(hw, dict(case, seed=case["seed"] + 10 * a), math="bf16x3", capacity=cap, replay="per", per_weighted_loss=True)
                   for a in keep}
        pop = hw.PopulationSAC(n, case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", capacity=cap, max_batch=B, math="bf16x3",
                               seed=seed, replay="per", per_weighted_loss=True)
        tabs = tables([rows] * n, ["halfnormal", "lognormal3", "floor1pct", "halfnormal", "fresh", "halfnormal", "lognormal3", "halfnormal"], 120)
        data = []
        for a in range(n):
            d = cases.per_transitions(dict(n=rows, obs=case["obs"], act=case["act"], seed=130 + a))
            d = {k: np.asarray(v, np.float32) for k, v in d.items()}
            data.append(d)
            pop.push_many(a, d["s"], d["a"], d["r"], d["s2"], d["d"])
            pop.set_priorities(a, *tabs[a])
            if a in singles:
                agent = singles[a][0]
                import_nets(hw, pop, a, agent)
                agent.replay_buffer.push_many(d["s"], d["a"], d["r"], d["s2"], d["d"])
                agent.replay_buffer.set_priorities(*tabs[a])
        rng = np.random.RandomState(5)
        e_next = rng.standard_normal((n, B, case["act"])).astype(np.float32)
        e_cur = rng.standard_normal((n, B, case["act"])).astype(np.float32)
        idx, w = sample_all(hw, pop, B)      # device-drawn uniforms
        u = [device_uniforms(agent_key(seed, a), 1, B) for a in range(n)]
        for a in range(n):
            ref_idx, ref_w = PO.sample(tabs[a][1], u[a], PO.beta(1))
            np.testing.assert_array_equal(idx[a], ref_idx, err_msg=f"agent {a}")
            assert ulp_diff(w[a], ref_w).max() <= 16, a
        N.check(lib.sacb_update(pop._h, B, None, N.ptr(e_next), N.ptr(e_cur), None, N.NO_LOSS_READBACK | N.USE_LAST_SAMPLE | N.WRITE_BACK_TD))
        losses = np.zeros((n, 3), np.float32)
        N.check(lib.sacb_get_losses_all(pop._h, N.ptr(losses)))
        assert np.isfinite(losses).all()
        for a, (agent, _) in singles.items():
            ref = agent.update_parameters(B, u=u[a], eps=(e_next[a], e_cur[a]))
            np.testing.assert_array_equal(losses[a], np.array([ref["q1_loss"], ref["q2_loss"], ref["policy_loss"]], np.float32), err_msg=f"agent {a}")
            assert_same_learner(pop, a, agent, "c2")
        # agent 0 against the oracle with the IS weights of its sample
        st = singles[0][1]
        b = {k: data[0][k][idx[0]] for k in ("s", "a", "r", "s2", "d")}
        b.update(eps_next=e_next[0], eps_cur=e_cur[0])
        ref, _ = oracle_step(None, st, case, b, hint=relu_hint(pop, case, agent_index=0), per_weights=w[0])
        check_losses({"q1_loss": losses[0, 0], "q2_loss": losses[0, 1], "policy_loss": losses[0, 2]}, ref, "c2 agent 0")
        check_state(population_state(pop, 0), st)
    finally:
        hw.use_networks("model1")


# ---- 8. refusals ---------------------------------------------------------------------------------------------------------------------
def test_refusals(hw):
    N = hw._native
    lib = N.lib()
    pop = per_pop(hw, 2, 1000, 32)
    push_zero_rows(hw, pop._h, 0, 100)
    push_zero_rows(hw, pop._h, 1, 20)      # fewer than B
    with pytest.raises(ValueError):
        pop.update_parameters(32)
    with pytest.raises(ValueError):
        sample_all(hw, pop, 32)
    with pytest.raises(ValueError):      # population sampling draws B rows from every agent: no idx hook
        pop.update_parameters(16, idx=np.zeros((2, 16), np.int64))
    push_zero_rows(hw, pop._h, 1, 20)
    sample_all(hw, pop, 32)
    # agent index out of range
    for bad in (-1, 2):
        with pytest.raises(ValueError):
            pop.priorities(bad)
        with pytest.raises(ValueError):
            N.check(lib.sacb_per_sample(pop._h, bad, None, 8, None, None, None, None, None, None, None))
        with pytest.raises(ValueError):
            N.check(lib.sacb_per_set_frame(pop._h, bad, 5))
        with pytest.raises(ValueError):
            N.check(lib.sacb_per_update_from_td(pop._h, bad, 8))
    # the pipelined step and K-step calls serve single-agent handles
    with pytest.raises(ValueError):
        N.check(lib.sacb_per_step(pop._h, 32, None, N.NO_LOSS_READBACK))
    with pytest.raises(ValueError):
        N.check(lib.sacb_update_steps(pop._h, 32, 2, None, N.NO_LOSS_READBACK))
    # capacity above the tail-free sampler form
    with pytest.raises(ValueError):
        per_pop(hw, 2, 2096129, 32)
    del pop
    big = per_pop(hw, 2, 2096128, 32)      # the largest accepted capacity
    del big
    # LayerNorm populations
    cfg = N.default_config()
    cfg.obs_dim, cfg.act_dim, cfg.hidden_dim, cfg.n_agents, cfg.capacity, cfg.replay_kind, cfg.layer_norm = 3, 2, 16, 2, 1000, N.REPLAY_PER, 1
    with pytest.raises(ValueError):
        N.create(cfg)
    # the per-agent accessors need replay="per"
    uni = hw.PopulationSAC(2, 3, 2, hidden_dim=16, device="cuda", capacity=100, max_batch=16)
    with pytest.raises(ValueError):
        uni.priorities(0)


# ---- 9. exploit leaves replay with its agent ----------------------------------------------------------------------------------------------------
def test_exploit_keeps_priorities_with_the_agent(hw):
    pop = per_pop(hw, 2, 5000, 64)
    tabs = tables([3000, 1200], ["halfnormal", "lognormal3"], 150)
    for a, (pri, pa) in enumerate(tabs):
        push_zero_rows(hw, pop._h, a, len(pri))
        pop.set_priorities(a, pri, pa)
    pop.set_frame(1, 77)
    before = (pop.priorities(1), pop.buffer_len(1), pop.frame(1))
    pop.exploit([1], [0])
    pop.synchronize()
    np.testing.assert_array_equal(pop.priorities(1), before[0])
    assert (pop.buffer_len(1), pop.frame(1)) == before[1:]
    np.testing.assert_array_equal(pop.priorities(0)[:3000], tabs[0][0])
