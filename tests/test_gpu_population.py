"""The benchmarked population (BASELINE.json configs[4]: 128 Humanoid agents of obs 348, act 17, three hidden layers of 512, B = 256)
against the oracle, and the device's random draws against a host restatement.

A. CPU: Philox4x32-10, philox_normal and draw_position (sample.cuh, tasks.cuh) restated in numpy; the restatement reproduces the
   Random123 known answers, its normals are N(0, 1) and its draws are permutations.
C. 128 agents with oracle weights, host positions and noise: selected agents against the oracle after each of two steps.
D. Production mode (positions and noise drawn on the device): every agent's positions equal the host restatement's, selected agents
   agree with an oracle step on the restated draws, and select_action_batch agrees with the oracle in all three modes.

The selected agents are 0, 1, the last one, and the first ones whose arena lies more than 2^31 and 2^32 bytes past agent 0's: the
agent offset of every pointer the update resolves is 64-bit there.  The bitwise comparison of the same population with single agents
is tests/test_gpu_sharded.py::test_population_stream_program_equals_single_agents."""
import ctypes
import gc

import numpy as np
import pytest
import scipy.stats

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.util import check_losses, check_state, oracle_step, population_state, relu_hint, selected_agents

C2 = cases.UPDATE_CASES["c2_humanoid_m2"]
M32 = np.uint64(0xFFFFFFFF)


# ---- host restatement of the device RNG ---------------------------------------------------------------------------------------
def philox4x32(c, k0, k1):
    """Philox4x32-10 exactly as sample.cuh's philox4x32: c = four uint32 counter words (scalars or arrays), key (k0, k1).
    uint64 arithmetic masked to 32 bits; a 32 x 32-bit product fits in 64 bits, so its high word is exact."""
    c = [np.asarray(x, np.uint64) for x in c]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def philox_normal(seed, stream, step, row, col):
    """sample.cuh's philox_normal: Box-Muller on the two top-24-bit uniforms of counter (row, col, step, stream).  The uniforms are
    formed in fp32 as on the device; logf / cospif are taken in float64, so a result can differ from the device's by a few ulp."""
    row, col, step, stream = np.broadcast_arrays(*(np.asarray(x, np.uint64) for x in (row, col, step, stream)))
    c = philox4x32([row, col, step, stream], int(seed) & 0xFFFFFFFF, int(seed) >> 32)
    u1 = ((c[0] >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)
    u2 = ((c[1] >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)
    two_u2 = np.float32(2.0) * u2
    return (np.sqrt(-2.0 * np.log(u1.astype(np.float64))) * np.cos(np.pi * two_u2.astype(np.float64))).astype(np.float32)


def draw_position(b, n, seed, agent, step):
    """tasks.cuh's draw_position for the rows `b` (an array): keyed bijection of [0, 2^bits) walked back into [0, n)."""
    s0, s1 = int(seed) & 0xFFFFFFFF, int(seed) >> 32
    key = [int(x) for x in philox4x32([step, agent, 0x1d5a7b1e, 0], s0, s1)]
    k2 = [int(x) for x in philox4x32([step, agent, 0x1d5a7b1f, 1], s0, s1)]
    bits = 1 if n <= 2 else (int(n) - 1).bit_length()
    mask = np.uint64(0xFFFFFFFF if bits >= 32 else (1 << bits) - 1)
    sh = np.uint64(max(1, bits // 2))

    def rounds(x):
        for r in range(4):
            x = (x * np.uint64(key[r] | 1) + np.uint64(k2[r])) & mask
            x ^= x >> sh
        return x
    x = rounds(np.asarray(b, np.uint64).copy())
    out = x >= np.uint64(n)
    while out.any():
        x[out] = rounds(x[out])
        out = x >= np.uint64(n)
    return x.astype(np.int64)


# ---- A. the restatement ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(ctr, key, want):
    """The Philox4x32-10 known-answer vectors of Random123 (kat_vectors)."""
    assert [int(x) for x in philox4x32(ctr, *key)] == want


def test_philox_normal_is_standard_normal():
    """2^20 draws over (row, col, step, stream) from one seed: Kolmogorov-Smirnov against N(0, 1), mean and variance within five
    standard errors of 0 and 1, and two streams at the same (row, col, step) uncorrelated."""
    seed = 0x0123456789ABCDEF
    row, col, step, stream = np.meshgrid(np.arange(256), np.arange(16), np.arange(16), np.arange(16), indexing="ij")
    z = philox_normal(seed, stream, step, row, col).astype(np.float64)
    n = z.size
    assert n == 1 << 20 and np.isfinite(z).all()
    assert scipy.stats.kstest(z.ravel(), "norm").pvalue > 1e-3
    assert abs(z.mean()) < 5 / np.sqrt(n), z.mean()
    assert abs(z.var() - 1) < 5 * np.sqrt(2 / n), z.var()
    a, b = z[..., 0].ravel(), z[..., 1].ravel()      # streams 0 and 1
    assert abs(np.corrcoef(a, b)[0, 1]) < 5 / np.sqrt(a.size)


@pytest.mark.parametrize("n", [1, 2, 3, 255, 256, 257, 100_000, (1 << 20) + 1])
def test_draw_position_is_a_permutation(n):
    """draw_position(., n) maps [0, n) onto itself one to one (cycle-walking included); other (agent, step) keys give other
    permutations."""
    seed = 0x5EEDF00DCAFE1234
    b = np.arange(n)
    perms = {}
    for agent, step in ((0, 0), (1, 0), (0, 1), (127, 7)):
        p = draw_position(b, n, seed, agent, step)
        np.testing.assert_array_equal(np.sort(p), b, err_msg=f"n={n} agent={agent} step={step}")
        perms[(agent, step)] = p
    if n >= 255:
        keys = list(perms)
        for i in range(len(keys)):
            for j in range(i + 1, len(keys)):
                assert not np.array_equal(perms[keys[i]], perms[keys[j]]), (n, keys[i], keys[j])


# ---- GPU helpers ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    hw.use_networks("model2")
    yield hw
    hw.use_networks("model1")


def load_oracle_agents(pop, case, seed0, keep):
    """Every agent i gets the weights of O.make_state(seed = seed0 + i); the oracle states of the agents in `keep` are returned."""
    states = {}
    for i in range(len(pop)):
        st = O.make_state(case["obs"], case["act"], case["hidden"], case["n_hidden"], seed=seed0 + i, head_scale=case["head_scale"])
        pop.load_agent(i, {**{f"{net}_state_dict": getattr(st, net) for net in ("policy", "q1", "q2", "q1_target", "q2_target")}, "alpha": st.alpha})
        if i in keep:
            states[i] = st
    return states


def agent_data(case, n_rows, agent, seed0):
    return O.make_batch(case["obs"], case["act"], n_rows, seed=seed0 + agent)


# ---- C. 128 agents, host positions and noise, against the oracle ------------------------------------------------------------------
@pytest.mark.gpu
def test_population_c2_128_matches_oracle(hw):
    """C2 x 128 with oracle weights (head_scale keeps the tanh unsaturated) and distinct data per agent, two steps on host positions
    and noise: after each step every selected agent's losses and whole state (nets, targets, Adam moments and steps, alpha) agree
    with the oracle, the oracle using that agent's ReLU masks (no disagreement outside the rounding band)."""
    case, n, B, rows = C2, 128, C2["batch"], 400
    pop = hw.PopulationSAC(n, case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", capacity=512, max_batch=B, seed=11)
    sel = selected_agents(pop, require_far=True)
    states = load_oracle_agents(pop, case, 3000, sel)
    data = {}
    for i in range(n):
        d = agent_data(case, rows, i, 4000)
        pop.push_many(i, d["s"], d["a"], d["r"], d["s2"], d["d"])
        if i in states:
            data[i] = d
    rng = np.random.RandomState(12)
    for step in range(2):
        idx = np.stack([rng.permutation(rows)[:B] for _ in range(n)]).astype(np.int64)
        e_next = rng.standard_normal((n, B, case["act"])).astype(np.float32)
        e_cur = rng.standard_normal((n, B, case["act"])).astype(np.float32)
        got = pop.update_parameters(B, idx=idx, eps=(e_next, e_cur))
        assert all(np.isfinite(list(g.values())).all() for g in got)
        for i, st in states.items():
            b = {k: data[i][k][idx[i]] for k in ("s", "a", "r", "s2", "d")}
            b.update(eps_next=e_next[i], eps_cur=e_cur[i])
            ref, _ = oracle_step(None, st, case, b, hint=relu_hint(pop, case, agent_index=i))
            check_losses(got[i], ref, (step, i))
            check_state(population_state(pop, i), st)
    del pop
    gc.collect()


# ---- D. production mode -----------------------------------------------------------------------------------------------------------
def ring_rows(d, n_pushed, capacity):
    """Transition arrays indexed by ring slot after `n_pushed` rows went into a ring of `capacity` in order."""
    pushed = np.arange(n_pushed)
    owner = np.empty(min(n_pushed, capacity), np.int64)
    owner[pushed[-capacity:] % capacity] = pushed[-capacity:]
    return {k: d[k][owner] for k in ("s", "a", "r", "s2", "d")}


@pytest.mark.gpu
@pytest.mark.parametrize("n,capacity", [(128, 100_000), (45, 1024)])
def test_population_production_draws_match_host(hw, n, capacity):
    """update_parameters(B) with no idx / eps, twice, 1300 distinct rows per agent: at 128 x 100 000 the ring offsets of the benchmark
    (agent 127's ring starts about 8.5e9 floats in), at 45 x 1024 every ring has wrapped (head != 0).

    * every agent's positions equal the host draw_position for (len, head, seed, agent, step), exactly;
    * each selected agent agrees with an oracle step on the rows at those positions, with noise eps_next[j] =
      philox_normal(seed, agent, step, j, .) and eps_cur[j] = philox_normal(seed, agent, step, B + j, .).  The host normals can
      differ from the device's by a few ulp of logf / cospif, far inside the loss and state budgets;
    * at 128 agents, select_action_batch agrees with O.select_action for every agent: evaluate, given eps, and device noise (stream
      0x5e1ec7, counter = the act_counter before the call, row = agent)."""
    N = hw._native
    lib = N.lib()
    case, B, n_rows = C2, C2["batch"], 1300
    pop = hw.PopulationSAC(n, case["obs"], case["act"], hidden_dim=case["hidden"], device="cuda", capacity=capacity, max_batch=B,
                           seed=0x5A5A00C0FFEE + n)
    seed = int(pop._cfg.seed)
    sel = selected_agents(pop, require_far=(n == 128))
    states = load_oracle_agents(pop, case, 5000, sel)
    ring = {}
    for i in range(n):
        d = agent_data(case, n_rows, i, 6000)
        pop.push_many(i, d["s"], d["a"], d["r"], d["s2"], d["d"])
        if i in states:
            ring[i] = ring_rows(d, n_rows, capacity)
    length, head = min(n_rows, capacity), (n_rows % capacity if n_rows > capacity else 0)
    assert all(pop.buffer_len(i) == length for i in (0, n - 1))
    slots = np.empty(B, np.int32)
    for _ in range(2):
        sc = N.Scalars()
        N.check(lib.sacb_get_scalars(pop._h, 0, ctypes.byref(sc)))
        step = int(sc.n_updates)
        got = pop.update_parameters(B)
        want = {}
        for i in range(n):
            N.check(lib.sacb_debug_read_slots(pop._h, i, N.ptr(slots, ctypes.c_int32), B))
            want[i] = (head + draw_position(np.arange(B), length, seed, i, step)) % capacity
            np.testing.assert_array_equal(slots, want[i], err_msg=f"agent {i} step {step}")
        for i, st in states.items():
            eps = philox_normal(seed, i, step, np.arange(2 * B)[:, None], np.arange(case["act"])[None, :])
            b = {k: v[want[i]] for k, v in ring[i].items()}
            b.update(eps_next=eps[:B], eps_cur=eps[B:])
            ref, _ = oracle_step(None, st, case, b, hint=relu_hint(pop, case, agent_index=i))
            check_losses(got[i], ref, (step, i))
            check_state(population_state(pop, i), st)
    if n == 128:
        rng = np.random.RandomState(13)
        obs = rng.standard_normal((n, case["obs"])).astype(np.float32)
        eps = rng.standard_normal((n, case["act"])).astype(np.float32)
        pol = [population_state(pop, i)["policy"] for i in range(n)]
        st = O.make_state(case["obs"], case["act"], case["hidden"], case["n_hidden"], seed=0)

        def ref_actions(evaluate, e):
            out = []
            for i in range(n):
                st.policy = pol[i]
                out.append(O.select_action(st, obs[i], evaluate=evaluate, eps=None if e is None else e[i]))
            return np.stack(out)
        np.testing.assert_allclose(pop.select_action(obs, evaluate=True), ref_actions(True, None), rtol=1e-3, atol=2e-5)
        np.testing.assert_allclose(pop.select_action(obs, eps=eps), ref_actions(False, eps), rtol=1e-3, atol=2e-5)
        sc = N.Scalars()
        N.check(lib.sacb_get_scalars(pop._h, 0, ctypes.byref(sc)))
        device_eps = philox_normal(seed, 0x5e1ec7, int(sc.act_counter), np.arange(n)[:, None], np.arange(case["act"])[None, :])
        np.testing.assert_allclose(pop.select_action(obs), ref_actions(False, device_eps), rtol=1e-3, atol=2e-5)
    del pop
    gc.collect()
