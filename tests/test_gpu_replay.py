"""GPU parity of the replay buffers through the C ABI: bit-exact for indices, priorities and stored rows.
Reference: replay_buffer.py:5-22 (uniform deque) and :25-90 (prioritized)."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import per_oracle as PO
from tests.golden import cases
from tests.test_oracle_per_golden import ulp_diff

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def filled_per(hw, case, bulk):
    tr = cases.per_transitions(case)
    buf = hw.PrioritizedReplayBuffer(case["capacity"])
    if bulk:
        for lo in range(0, case["n"], 700):      # odd chunking: exercises ring wrap inside a bulk push
            hi = min(case["n"], lo + 700)
            buf.push_many(tr["s"][lo:hi], tr["a"][lo:hi], tr["r"][lo:hi], tr["s2"][lo:hi], tr["d"][lo:hi])
    else:
        for i in range(case["n"]):
            buf.push(tr["s"][i], tr["a"][i], tr["r"][i], tr["s2"][i], bool(tr["d"][i]))
    return buf, tr


@pytest.mark.parametrize("name", list(cases.PER_CASES))
def test_per_matches_reference_golden(hw, name):
    case = cases.PER_CASES[name]
    g = np.load(os.path.join(GOLD, f"per_{name}.npz"))
    buf, tr = filled_per(hw, case, bulk=case["n"] > 2000)
    assert len(buf) == min(case["n"], case["capacity"])
    np.testing.assert_array_equal(buf.priorities, g["prio_after_push"])          # max-priority rule, :38
    assert buf.pos == int(g["pos_after_push"])
    m = min(case["n"], case["capacity"])
    pri = np.zeros(case["capacity"], np.float32)
    pri[:m] = cases.per_priorities(case)[:m]
    pa = np.zeros(case["capacity"], np.float32)
    pa[:m] = g["p_alpha"]                                                       # numpy's own p**alpha (ISA dependent)
    buf.set_priorities(pri, pa)
    k = min(case["batch"], m)
    for call in range(case["calls"]):
        u = PO.uniform_draws(case["seed"] * 10 + call, k)
        s, a, r, s2, d, idx, w = buf.sample(case["batch"], u=u)
        np.testing.assert_array_equal(idx, g["idx"][call])                       # BIT-EXACT indices
        assert ulp_diff(w, g["weights"][call]).max() <= 16                       # two float32 pow + divide by the max
        if call == 0:
            np.testing.assert_array_equal(r, g["sample0/r"])
            np.testing.assert_array_equal(s, g["sample0/s"])
            np.testing.assert_array_equal(d, g["sample0/d"])
    assert buf.frame == 1 + case["calls"]
    buf.update_priorities(g["upd_idx"], torch.from_numpy(cases.per_td(case)[: g["upd_idx"].size]))
    np.testing.assert_array_equal(buf.priorities, g["prio_after_update"])        # BIT-EXACT priorities, last duplicate wins
    buf.push(tr["s"][0], tr["a"][0], tr["r"][0], tr["s2"][0], False)
    np.testing.assert_array_equal(buf.priorities, g["prio_after_push2"])
    assert buf.pos == int(g["pos_after_push2"])


# Above 2 096 128 rows the chunk prefixes do not fit into shared memory: the 2.5 M case runs the sampler form with last-CTA tails
# (per_sum with its tail -> per_chunk -> per_search), every other size the tail-free form.
@pytest.mark.parametrize("dist,n", [("halfnormal", 100003), ("floor1pct", 250000), ("lognormal3", 1000000), ("halfnormal", 1000000), ("fresh", 1000000),
                                    ("halfnormal", 2500000)])
def test_per_bit_exact_vs_oracle_large(hw, dist, n):
    """BASELINE.json sizes (up to 1 M): indices bit-exact against the C oracle on the same p**alpha table,
    including the adversarial priority sets of SURVEY H6.4 that defeat a naive parallel scan."""
    case = dict(n=n, capacity=n, batch=256, seed=31, dist=dist)
    rng = np.random.RandomState(9)
    buf = hw.PrioritizedReplayBuffer(n)
    buf.push_many(rng.standard_normal((8, 2)), rng.standard_normal((8, 1)), np.zeros(8), rng.standard_normal((8, 2)), np.zeros(8))
    lib, N = hw._native.lib(), hw._native
    # fill the ring cheaply: only the tables matter for this test
    rows = np.zeros((n - 8, int(lib.sacb_row_floats(buf._h))), np.float32)
    N.check(lib.sacb_push_rows(buf._h, 0, N.ptr(rows), n - 8))
    pri = cases.per_priorities(case)
    pa = (pri ** np.float32(0.6)).astype(np.float32)
    buf.set_priorities(pri, pa)
    assert PO.pairwise_sum(pa) == pa.sum()
    for call in range(3):
        u = rng.random_sample(256)
        *_, idx, w = buf.sample(256, u=u)
        ref_idx, ref_w = PO.sample(pa, u, PO.beta(1 + call))
        np.testing.assert_array_equal(idx, ref_idx)
        assert ulp_diff(w, ref_w).max() <= 16
    st = buf._stats()
    assert st.total_f32 == pa.sum()                                              # numpy pairwise tree reproduced exactly
    # device powf vs numpy's: documented <= 2 ulp (SURVEY H6.3)
    buf.set_priorities(pri)
    *_, idx2, _ = buf.sample(256, u=u)
    assert np.mean(idx2 == ref_idx) > 0.99


# 2.5 M rows: above 2 096 128 the chunk prefixes do not fit into shared memory, so this case runs the form with last-CTA tails
@pytest.mark.parametrize("dist,n", [("lognormal3", 50000), ("halfnormal", 1000000), ("floor1pct", 300000), ("lognormal3", 1000000),
                                    ("floor1pct", 2500000)])
def test_per_ambiguous_samples_take_the_exact_path(hw, dist, n):
    """u placed exactly ON cdf boundaries: the certified fast path must flag them and the exact sequential evaluation decides
    (chunks without fine elements and without a binade crossing are jumped, the others are walked element by element)."""
    case = dict(n=n, capacity=n, batch=256, seed=41, dist=dist)     # tiny probabilities: bits below 2^-52 ("fine" elements)
    pri = cases.per_priorities(case)
    pa = (pri ** np.float32(0.6)).astype(np.float32)
    buf = hw.PrioritizedReplayBuffer(n)
    lib, N = hw._native.lib(), hw._native
    buf.push_many(np.zeros((1, 2)), np.zeros((1, 1)), np.zeros(1), np.zeros((1, 2)), np.zeros(1))
    rows = np.zeros((n - 1, int(lib.sacb_row_floats(buf._h))), np.float32)
    N.check(lib.sacb_push_rows(buf._h, 0, N.ptr(rows), n - 1))
    buf.set_priorities(pri, pa)
    _, _, _, cdf = PO.sample(pa, np.array([0.5]), 0.4, want_tables=True)
    pick = np.random.RandomState(1).randint(0, n - 1, 256)
    u = cdf[pick].copy()
    u[::2] = np.nextafter(u[::2], 0.0)
    *_, idx, _ = buf.sample(256, u=u)
    ref_idx, _ = PO.sample(pa, u, 0.4)
    np.testing.assert_array_equal(idx, ref_idx)
    st = buf._stats()
    assert st.n_fine > 0 and st.n_flagged > 0 and st.n_exact_fallbacks >= 1, (st.n_fine, st.n_flagged, st.n_exact_fallbacks)


@pytest.mark.parametrize("name", list(cases.UNIFORM_CASES))
def test_uniform_buffer_matches_reference_golden(hw, name):
    case = cases.UNIFORM_CASES[name]
    g = np.load(os.path.join(GOLD, f"uniform_{name}.npz"))
    buf = hw.ReplayBuffer(case["capacity"])
    for i in range(case["n"]):
        buf.push(np.full(3, i, np.float32), np.full(2, -i, np.float32), float(i), np.full(3, i + 0.5, np.float32), i % 5 == 0)
    assert len(buf) == int(g["len"])
    random.seed(case["seed"])
    for call in range(case["calls"]):
        s, a, r, s2, d = buf.sample(case["batch"])
        np.testing.assert_array_equal(r.astype(np.int64), g["r_ids"][call])     # same picks as random.sample(deque, k)
        if call == 0:
            np.testing.assert_array_equal(s, g["s"])
            np.testing.assert_array_equal(a, g["a"])
            np.testing.assert_array_equal(s2, g["s2"])
            np.testing.assert_array_equal(d.astype(bool), g["d"])
    with pytest.raises(ValueError):
        buf.sample(len(buf) + 1)                                                 # random.sample's error


def test_buffer_attribute_round_trip(hw):
    buf = hw.ReplayBuffer(50)
    for i in range(70):
        buf.push(np.full(4, i), np.full(2, i), i, np.full(4, i + 1), i % 3 == 0)
    dq = buf.buffer
    assert len(dq) == 50 and dq.maxlen == 50 and dq[0][2] == 20.0 and dq[-1][2] == 69.0 and dq[1][4] is True
    other = hw.ReplayBuffer(50)
    other.buffer = dq
    assert len(other) == 50 and other.buffer[7][2] == dq[7][2]


def test_uniform_sample_larger_than_the_device_staging_area(hw):
    """replay_buffer.py:12-17 takes any batch size up to len(buffer); the library gathers through a staging area of 4096 rows."""
    n, obs, act = 6000, 5, 2
    rng = np.random.RandomState(4)
    s, a, s2 = rng.randn(n, obs).astype(np.float32), rng.randn(n, act).astype(np.float32), rng.randn(n, obs).astype(np.float32)
    r, d = rng.randn(n).astype(np.float32), (rng.rand(n) < 0.1).astype(np.float32)
    buf = hw.ReplayBuffer(8192)
    buf.push_many(s, a, r, s2, d)
    random.seed(11)
    expect = np.asarray(random.sample(range(n), 5000))
    random.seed(11)
    gs, ga, gr, gs2, gd = buf.sample(5000)
    np.testing.assert_array_equal(gs, s[expect]); np.testing.assert_array_equal(ga, a[expect]); np.testing.assert_array_equal(gr, r[expect])
    np.testing.assert_array_equal(gs2, s2[expect]); np.testing.assert_array_equal(gd, d[expect])
    per = hw.PrioritizedReplayBuffer(8192)
    per.push_many(s, a, r, s2, d)
    with pytest.raises(ValueError):
        per.sample(5000)


@pytest.mark.parametrize("launch", ["staged", "persistent"])
def test_pipelined_step_equals_sequential(hw, launch):
    """sacb_per_step (write-back + next sample on a second stream under the tail of the update) == the three calls in sequence, bitwise.
    (persistent launch mode: the single cooperative launch cannot be split, the PER work simply follows it on the second stream)"""
    import ctypes
    import torch
    from tests.util import make_agent
    N = hw._native
    lib = N.lib()
    case = cases.UPDATE_CASES["tiny_m2"]
    B, n, cap = case["batch"], 3000, 4096
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
    seq, pipe = agents
    steps = 7
    for _ in range(steps):
        N.check(lib.sacb_per_sample(seq._h, 0, None, B, None, None, None, None, None, None, None))
        N.check(lib.sacb_update(seq._h, B, None, None, None, None, N.USE_LAST_SAMPLE | N.NO_LOSS_READBACK))
        N.check(lib.sacb_per_update_from_td(seq._h, 0, B))
    for _ in range(steps):
        pipe.learner_step(B)
    seq.synchronize(); pipe.synchronize()
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        a, b = getattr(seq, net).state_dict(), getattr(pipe, net).state_dict()
        for k in a:
            assert torch.equal(a[k], b[k]), (net, k)
    pa, pb = np.empty(cap, np.float32), np.empty(cap, np.float32)
    N.check(lib.sacb_per_get_priorities(seq._h, 0, N.ptr(pa), cap))
    N.check(lib.sacb_per_get_priorities(pipe._h, 0, N.ptr(pb), cap))
    assert np.array_equal(pa, pb)
    assert not np.array_equal(pa, pri)      # the write-back happened
    la, lb = np.zeros(3, np.float32), np.zeros(3, np.float32)
    N.check(lib.sacb_get_losses(seq._h, 0, N.ptr(la))); N.check(lib.sacb_get_losses(pipe._h, 0, N.ptr(lb)))
    assert np.array_equal(la, lb) and np.all(np.isfinite(la))


@pytest.mark.parametrize("weighted", [True, False])
def test_update_parameters_equals_the_three_calls(hw, weighted):
    """update_parameters over the prioritized buffer (sample, then sacb_update with SACB_WRITE_BACK_TD: the |TD| write-back enqueued by the
    same call behind the loss copy) == sacb_per_sample / sacb_update / sacb_per_update_from_td in sequence, bitwise, with the trainer's
    push in front of every step, while the ring still grows and after it has filled up."""
    import ctypes
    import torch
    from tests.util import make_agent
    N = hw._native
    lib = N.lib()
    case = cases.UPDATE_CASES["tiny_m2"]
    B, n, cap, steps = case["batch"], 3040, 3072, 50
    rng = np.random.RandomState(11)
    S, A = rng.standard_normal((n + steps, case["obs"])).astype(np.float32), rng.uniform(-0.4, 0.4, (n + steps, case["act"])).astype(np.float32)
    R, S2 = rng.standard_normal(n + steps).astype(np.float32), rng.standard_normal((n + steps, case["obs"])).astype(np.float32)
    D = rng.uniform(size=n + steps) < 0.1
    pri = np.zeros(cap, np.float32)
    pri[:n] = np.abs(rng.standard_normal(n)) + 1e-6
    agents = []
    for _ in range(2):
        agent, _st = make_agent(hw, case, math="bf16x3", launch="staged", capacity=cap, replay="per", per_weighted_loss=weighted)
        agent.replay_buffer.push_many(S[:n], A[:n], R[:n], S2[:n], D[:n])
        agent.replay_buffer.set_priorities(pri)
        agents.append(agent)
    seq, one = agents
    for i in range(steps):
        u = rng.random_sample(B)
        t = n + i
        for a in agents:
            a.replay_buffer.push(S[t], A[t], float(R[t]), S2[t], bool(D[t]))
        seq.replay_buffer._flush()
        la = np.zeros(3, np.float32)
        N.check(lib.sacb_per_sample(seq._h, 0, N.ptr(u, ctypes.c_double), B, None, None, None, None, None, None, None))
        N.check(lib.sacb_update(seq._h, B, None, None, None, N.ptr(la), N.USE_LAST_SAMPLE))
        if weighted:
            N.check(lib.sacb_per_update_from_td(seq._h, 0, B))
        out = one.update_parameters(B, u=u)
        assert (float(la[0]), float(la[1]), float(la[2])) == (out["q1_loss"], out["q2_loss"], out["policy_loss"]), i
    seq.synchronize(); one.synchronize()
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        a, b = getattr(seq, net).state_dict(), getattr(one, net).state_dict()
        for k in a:
            assert torch.equal(a[k], b[k]), (net, k)
    pa, pb = np.empty(cap, np.float32), np.empty(cap, np.float32)
    N.check(lib.sacb_per_get_priorities(seq._h, 0, N.ptr(pa), cap))
    N.check(lib.sacb_per_get_priorities(one._h, 0, N.ptr(pb), cap))
    assert np.array_equal(pa, pb)
    assert weighted == (not np.array_equal(pa[100:n], pri[100:n]))      # (slots the pushes did not reach) the write-back happens exactly in the IS-weighted mode
    assert seq.replay_buffer.frame == one.replay_buffer.frame


def test_trainer_path_is_reproducible_over_many_steps(hw):
    """1500 trainer steps (push + update_parameters, host uniforms, losses read back) on two handles fed the same data: identical
    losses at every step and identical weights / priorities at the end.  The pushed row, the uniforms and the losses cross the bus
    through pinned blocks that the kernels touch directly and the host reuses every step: a reuse before the device is done with a
    block would show up here as a difference."""
    import torch
    from tests.util import make_agent
    N = hw._native
    lib = N.lib()
    case = cases.UPDATE_CASES["tiny_m2"]
    B, n, cap, steps = case["batch"], 2000, 2048, 1500
    rng = np.random.RandomState(23)
    S, A = rng.standard_normal((n, case["obs"])).astype(np.float32), rng.uniform(-0.4, 0.4, (n, case["act"])).astype(np.float32)
    R, S2, D = rng.standard_normal(n).astype(np.float32), rng.standard_normal((n, case["obs"])).astype(np.float32), rng.uniform(size=n) < 0.1
    agents = []
    for _ in range(2):
        agent, _st = make_agent(hw, case, math="bf16x3", launch="staged", capacity=cap, replay="per", per_weighted_loss=True)
        agent.replay_buffer.push_many(S, A, R, S2, D)
        agents.append(agent)
    a0, a1 = agents
    for i in range(steps):
        u = rng.random_sample(B)
        s, a, r, s2, d = rng.standard_normal(case["obs"]), rng.uniform(-0.4, 0.4, case["act"]), float(rng.standard_normal()), rng.standard_normal(case["obs"]), bool(rng.uniform() < 0.1)
        outs = []
        for ag in agents:
            ag.replay_buffer.push(s, a, r, s2, d)
            outs.append(ag.update_parameters(B, u=u))
        assert outs[0] == outs[1], i
        assert all(np.isfinite(v) for v in outs[0].values()), i
    a0.synchronize(); a1.synchronize()
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        x, y = getattr(a0, net).state_dict(), getattr(a1, net).state_dict()
        for k in x:
            assert torch.equal(x[k], y[k]), (net, k)
    pa, pb = np.empty(cap, np.float32), np.empty(cap, np.float32)
    N.check(lib.sacb_per_get_priorities(a0._h, 0, N.ptr(pa), cap))
    N.check(lib.sacb_per_get_priorities(a1._h, 0, N.ptr(pb), cap))
    assert np.array_equal(pa, pb)


@pytest.mark.parametrize("dist,n", [("floor1pct", 1000000), ("lognormal3", 1000000)])
def test_per_many_calls_on_adversarial_priorities(hw, dist, n):
    """120 sample() calls (30 720 draws) on the priority sets with thousands of fine probabilities: every index equals numpy's, whether the
    sample was certified on the fast path (window = (12 F + 8) eps / last, replay.cu) or went through the exact pass."""
    case = dict(n=n, capacity=n, batch=256, seed=51, dist=dist)
    pri = cases.per_priorities(case)
    pa = (pri ** np.float32(0.6)).astype(np.float32)
    buf = hw.PrioritizedReplayBuffer(n)
    lib, N = hw._native.lib(), hw._native
    buf.push_many(np.zeros((1, 2)), np.zeros((1, 1)), np.zeros(1), np.zeros((1, 2)), np.zeros(1))
    rows = np.zeros((n - 1, int(lib.sacb_row_floats(buf._h))), np.float32)
    N.check(lib.sacb_push_rows(buf._h, 0, N.ptr(rows), n - 1))
    buf.set_priorities(pri, pa)
    rng = np.random.RandomState(7)
    for call in range(120):
        u = rng.random_sample(256)
        *_, idx, _ = buf.sample(256, u=u)
        ref_idx, _ = PO.sample(pa, u, PO.beta(1 + call))
        np.testing.assert_array_equal(idx, ref_idx, err_msg=f"call {call}")
    st = buf._stats()
    assert st.n_fine > 500, st.n_fine      # the case really is adversarial (floor probabilities below 2^-28 only appear at N = 1 M)
