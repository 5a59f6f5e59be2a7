"""GPU tests of the two sharded modes on ONE device (SURVEY 4.4 / 8e): a population of independent agents in one
handle must equal the same agents run one by one, and the data-parallel step over two logical shards must equal the
single-agent step on the concatenated batch."""
import ctypes
import gc

import numpy as np
import pytest
import torch

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.util import batch_of, make_agent, net_params, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    return hw


def _push_all(agent, b):
    agent.replay_buffer.push_many(b["s"], b["a"], b["r"], b["s2"], b["d"])


def test_population_equals_independent_agents(hw):
    """BASELINE.json configs[4] in miniature: 3 agents with distinct weights / data / eps in one handle (agent = grid
    dimension and 4th TMA coordinate) against three single-agent handles.  No communication exists to test."""
    N = hw._native
    lib = N.lib()
    case = cases.UPDATE_CASES["tiny_m2"]
    B, n_agents = case["batch"], 3
    singles, batches = [], []
    for a in range(n_agents):
        agent, _ = make_agent(hw, dict(case, seed=case["seed"] + 10 * a), math="bf16x3", capacity=64)
        b = batch_of(dict(case, seed=case["seed"] + 10 * a), 0)
        _push_all(agent, b)
        singles.append(agent)
        batches.append(b)
    cfg = N.default_config()
    c0 = singles[0]._cfg
    for f, _ in N.Config._fields_:
        if f != "reserved":
            setattr(cfg, f, getattr(c0, f))
    cfg.n_agents = n_agents
    h = N.create(cfg)
    try:
        nets = ("policy", "q1", "q2", "q1_target", "q2_target")
        for a, agent in enumerate(singles):
            for net_id, net in enumerate(nets):
                for t, (_, p) in enumerate(getattr(agent, net).named_parameters()):
                    host = N.f32(p.detach().cpu().numpy())
                    N.check(lib.sacb_import_tensor(h, a, net_id, N.SLOT_PARAM, t, N.ptr(host), host.size))
            b = batches[a]
            s, ac, r, s2, d = (N.f32(b[k]) for k in ("s", "a", "r", "s2", "d"))
            N.check(lib.sacb_push(h, a, N.ptr(s), N.ptr(ac), N.ptr(r), N.ptr(s2), N.ptr(d), B))
        idx = np.ascontiguousarray(np.tile(np.arange(B, dtype=np.int64), (n_agents, 1)))
        e_next = np.ascontiguousarray(np.stack([b["eps_next"] for b in batches]), np.float32)
        e_cur = np.ascontiguousarray(np.stack([b["eps_cur"] for b in batches]), np.float32)
        N.check(lib.sacb_update(h, B, N.ptr(idx, ctypes.c_int64), N.ptr(e_next), N.ptr(e_cur), None, N.NO_LOSS_READBACK))
        N.check(lib.sacb_synchronize(h))
        for a, agent in enumerate(singles):
            got = agent.update_parameters(B, idx=np.arange(B), eps=(batches[a]["eps_next"], batches[a]["eps_cur"]))
            losses = np.zeros(3, np.float32)
            N.check(lib.sacb_get_losses(h, a, N.ptr(losses)))
            np.testing.assert_array_equal(losses, np.array([got["q1_loss"], got["q2_loss"], got["policy_loss"]], np.float32))
            for net_id, net in enumerate(nets):
                for t, (nm, p) in enumerate(getattr(agent, net).named_parameters()):
                    out = np.empty(p.numel(), np.float32)
                    N.check(lib.sacb_export_tensor(h, a, net_id, N.SLOT_PARAM, t, N.ptr(out), out.size))
                    np.testing.assert_array_equal(out.reshape(p.shape), p.detach().cpu().numpy(), err_msg=f"agent {a} {net}.{nm}")
        # population select_action (SURVEY 8f rank 1): row i of the batch acts with agent i's policy, one chain of launches
        rng = np.random.RandomState(5)
        obs = rng.standard_normal((n_agents, case["obs"])).astype(np.float32)
        eps = rng.standard_normal((n_agents, case["act"])).astype(np.float32)
        for evaluate, e in ((1, None), (0, eps)):
            act = np.empty((n_agents, case["act"]), np.float32)
            N.check(lib.sacb_select_action_batch(h, N.ptr(obs), evaluate, N.ptr(e), N.ptr(act)))
            for a, agent in enumerate(singles):
                ref = agent.select_action(obs[a], evaluate=bool(evaluate), eps=None if e is None else e[a:a + 1])
                np.testing.assert_array_equal(act[a], ref, err_msg=f"agent {a} evaluate={evaluate}")
    finally:
        lib.sacb_destroy(h)


@pytest.mark.parametrize("name", ["tiny_m2", "c1_bipedal_m1"])
def test_data_parallel_two_shards_equal_full_batch(hw, name):
    """BASELINE.json configs[3] on one GPU: two replicas, half the batch each, gradient slabs averaged by hand exactly as
    the all-reduce would; result == the single-agent update on the whole batch up to fp32 reassociation of the batch sum."""
    N = hw._native
    lib = N.lib()
    case = cases.UPDATE_CASES[name]
    B = case["batch"]
    b = batch_of(case, 0)
    full, _ = make_agent(hw, case, math="bf16x3", capacity=1024)
    _push_all(full, b)
    ref = full.update_parameters(B, idx=np.arange(B), eps=(b["eps_next"], b["eps_cur"]))
    shards = []
    for r in range(2):
        ag, _ = make_agent(hw, case, math="bf16x3", capacity=1024)
        _push_all(ag, b)
        shards.append(hw.distributed.DataParallelSAC(ag))
    half = B // 2
    rows = [np.arange(0, half, dtype=np.int64), np.arange(half, B, dtype=np.int64)]
    for phase in (0, 1):
        for r, dp in enumerate(shards):
            ix = rows[r]
            e = (N.f32(b["eps_next"][ix]), N.f32(b["eps_cur"][ix]))
            N.check(lib.sacb_dp_backward(dp.agent._h, phase, half, N.ptr(ix, ctypes.c_int64) if phase == 0 else None, N.ptr(e[0]), N.ptr(e[1])))
            dp.agent.synchronize()
        for s0, s1 in zip(shards[0].gradient_slabs(phase), shards[1].gradient_slabs(phase)):      # what all-reduce(mean) does
            m = (s0 + s1) / 2
            s0.copy_(m); s1.copy_(m)
        torch.cuda.synchronize()
        for dp in shards:
            N.check(lib.sacb_dp_apply(dp.agent._h, phase))
            dp.agent.synchronize()
    lr = 3e-4
    for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
        want = net_params(full, net)
        for r in range(2):
            mine = net_params(shards[r].agent, net)
            for nm in want:
                # identical gradients up to reassociation; Adam's first step is sign-like, so a gradient within rounding of
                # zero may move by +lr in one run and -lr in the other: allow a handful of such elements
                bad = np.mean(np.abs(mine[nm] - want[nm]) > 0.02 * lr)
                assert bad < 5e-3, (net, nm, r, bad)
    np.testing.assert_array_equal(net_params(shards[0].agent, "q1")["fc1.weight"], net_params(shards[1].agent, "q1")["fc1.weight"])
    a_full, a_dp = float(torch.as_tensor(full.alpha).reshape(-1)[0]), float(torch.as_tensor(shards[0].agent.alpha).reshape(-1)[0])
    assert abs(a_full - a_dp) <= 1e-6 * abs(a_full)
    l0 = np.zeros(3, np.float32); l1 = np.zeros(3, np.float32)
    N.check(lib.sacb_get_losses(shards[0].agent._h, 0, N.ptr(l0))); N.check(lib.sacb_get_losses(shards[1].agent._h, 0, N.ptr(l1)))
    np.testing.assert_allclose((l0 + l1) / 2, [ref["q1_loss"], ref["q2_loss"], ref["policy_loss"]], rtol=2e-5)


def test_data_parallel_wrapper_world1_matches_plain_update(hw):
    """DataParallelSAC without a process group (world = 1) is the plain update: backward/export + apply kernels vs the fused epilogues."""
    case = cases.UPDATE_CASES["tiny_m1"]
    B = case["batch"]
    b = batch_of(case, 0)
    plain, _ = make_agent(hw, case, math="bf16x3", capacity=256)
    dp_agent, _ = make_agent(hw, case, math="bf16x3", capacity=256)
    _push_all(plain, b); _push_all(dp_agent, b)
    ref = plain.update_parameters(B, idx=np.arange(B), eps=(b["eps_next"], b["eps_cur"]))
    got = hw.distributed.DataParallelSAC(dp_agent).update_parameters(B, idx=np.arange(B), eps=(b["eps_next"], b["eps_cur"]))
    for k in ref:
        assert abs(got[k] - ref[k]) <= 1e-6 * abs(ref[k]) + 1e-7
    for net in ("policy", "q1", "q2", "q1_target"):
        w, m = net_params(plain, net), net_params(dp_agent, net)
        for nm in w:
            assert np.mean(np.abs(w[nm] - m[nm]) > 0.02 * 3e-4) < 5e-3, (net, nm)
    assert dp_agent.policy_optimizer.state_dict()["state"][0]["step"] == 1


def test_population_class_equals_seeded_single_agents(hw):
    """PopulationSAC(seeds=[..]) agent i == `torch.manual_seed(seeds[i]); SAC(...)`: same initial weights (reference initialiser
    calls in the order of sac_imp.py:28-36), and after two updates on the same rows / eps the same weights and losses, bitwise."""
    hw.use_networks("model2")
    obs, act, hid, B, seeds = 13, 5, 48, 24, [7, 3, 11]
    pop = hw.PopulationSAC(len(seeds), obs, act, hidden_dim=hid, device="cuda", seeds=seeds, capacity=64, max_batch=B, seed=99)
    singles = []
    rng = np.random.RandomState(0)
    data = []
    for i, sd in enumerate(seeds):
        torch.manual_seed(sd)
        ag = hw.SAC(obs, act, hidden_dim=hid, device="cuda", capacity=64, max_batch=B, seed=99)
        b = O.make_batch(obs, act, 40, seed=500 + i)
        ag.replay_buffer.push_many(b["s"], b["a"], b["r"], b["s2"], b["d"])
        pop.push_many(i, b["s"], b["a"], b["r"], b["s2"], b["d"])
        singles.append(ag)
        st = pop.agent_state(i)
        for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
            for k, v in net_params(ag, net).items():
                np.testing.assert_array_equal(st[f"{net}_state_dict"][k].numpy(), v, err_msg=f"initial weights agent {i} {net}.{k}")
    assert pop.buffer_len(1) == 40
    for step in range(2):
        idx = np.stack([rng.permutation(40)[:B] for _ in seeds]).astype(np.int64)
        e_next = rng.standard_normal((len(seeds), B, act)).astype(np.float32)
        e_cur = rng.standard_normal((len(seeds), B, act)).astype(np.float32)
        got = pop.update_parameters(B, idx=idx, eps=(e_next, e_cur))
        for i, ag in enumerate(singles):
            ref = ag.update_parameters(B, idx=idx[i], eps=(e_next[i], e_cur[i]))
            assert got[i] == ref, (step, i, got[i], ref)
    for i, ag in enumerate(singles):
        st = pop.agent_state(i)
        for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
            for k, v in net_params(ag, net).items():
                np.testing.assert_array_equal(st[f"{net}_state_dict"][k].numpy(), v, err_msg=f"agent {i} {net}.{k}")
        assert abs(float(st["alpha"]) - float(ag.alpha)) == 0.0
    # production mode: positions and eps drawn on the device, every agent its own stream
    out = pop.update_parameters(B)
    assert len(out) == len(seeds) and all(np.isfinite(list(o.values())).all() for o in out)
    assert out[0] != out[1]
    acts = pop.select_action(rng.standard_normal((len(seeds), obs)), evaluate=True)
    assert acts.shape == (len(seeds), act) and np.all(np.abs(acts) <= 0.4 + 1e-6)
    hw.use_networks("model1")


def test_device_index_draw_is_a_sample_without_replacement(hw):
    """SACB_DEVICE_INDICES: the gather stage draws B DISTINCT ring positions per update (random.sample semantics,
    replay_buffer.py:15), different every step, covering the ring uniformly; wrapped ring (head != 0) included."""
    N = hw._native
    lib = N.lib()
    hw.use_networks("model1")
    obs, act, B, cap = 6, 2, 64, 300
    agent = hw.SAC(obs, act, hidden_dim=16, device="cuda", capacity=cap, max_batch=B, seed=5)
    n = 420                                   # > capacity: the ring has wrapped
    ids = np.arange(n, dtype=np.float32)
    agent.replay_buffer.push_many(np.tile(ids[:, None], (1, obs)), np.zeros((n, act), np.float32), ids, np.tile(ids[:, None], (1, obs)), np.zeros(n))
    counts = np.zeros(n)
    seen = []
    slots = np.empty(B, np.int32)
    for step in range(200):
        N.check(lib.sacb_update(agent._h, B, None, None, None, None, N.NO_LOSS_READBACK | N.DEVICE_INDICES))
        N.check(lib.sacb_debug_read_slots(agent._h, 0, N.ptr(slots, ctypes.c_int32), B))
        assert len(set(slots.tolist())) == B and slots.min() >= 0 and slots.max() < cap
        seen.append(slots.copy())
        counts[slots] += 1
    assert not np.array_equal(seen[0], seen[1])
    hit = counts[:cap]
    assert hit.min() > 0 and abs(hit.mean() - 200 * B / cap) < 1e-9 and hit.std() < 3.5 * np.sqrt(200 * B / cap)      # ~Binomial spread
    with pytest.raises(ValueError):
        small = hw.SAC(obs, act, hidden_dim=16, device="cuda", capacity=cap, max_batch=B, seed=5)
        small.replay_buffer.push_many(np.zeros((10, obs)), np.zeros((10, act)), np.zeros(10), np.zeros((10, obs)), np.zeros(10))
        N.check(lib.sacb_update(small._h, B, None, None, None, None, N.NO_LOSS_READBACK | N.DEVICE_INDICES))


@pytest.mark.parametrize("replay", ["uniform", "per"])
def test_k_steps_per_call_equal_single_calls(hw, replay):
    """learner_steps(k=K) (sacb_update_steps: K steps enqueued back to back, ONE loss read-back) == K single calls, bitwise."""
    hw.use_networks("model1")
    obs, act, B, K = 11, 3, 32, 6
    agents = []
    rng = np.random.RandomState(1)
    b = O.make_batch(obs, act, 500, seed=77)
    pri = (np.abs(rng.standard_normal(512)) + 1e-6).astype(np.float32)
    for _ in range(2):
        torch.manual_seed(3)
        ag = hw.SAC(obs, act, hidden_dim=32, device="cuda", capacity=512, max_batch=B, seed=42, replay=replay, per_weighted_loss=(replay == "per"))
        ag.replay_buffer.push_many(b["s"], b["a"], b["r"], b["s2"], b["d"])
        if replay == "per":
            ag.replay_buffer.set_priorities(pri)
        agents.append(ag)
    many = agents[0].learner_steps(B, k=K)
    single = [agents[1].learner_steps(B, k=1)[0] for _ in range(K)]
    assert many == single
    for net in ("policy", "q1", "q2_target"):
        for k, v in net_params(agents[0], net).items():
            np.testing.assert_array_equal(v, net_params(agents[1], net)[k])
    if replay == "per":
        np.testing.assert_array_equal(agents[0].replay_buffer.priorities, agents[1].replay_buffer.priorities)


def _equal_states(got, want, tag):
    for k, v in want.items():
        if isinstance(v, dict):
            for nm in v:
                np.testing.assert_array_equal(got[k][nm], v[nm], err_msg=f"{tag} {k}.{nm}")
        elif isinstance(v, tuple):      # (step, m, v) of an optimizer
            assert got[k][0] == v[0], (tag, k, got[k][0], v[0])
            _equal_states({"m": got[k][1], "v": got[k][2]}, {"m": v[1], "v": v[2]}, f"{tag} {k}")
        else:
            assert got[k] == v, (tag, k, got[k], v)


def _n_tiles(hw, h):
    st = hw._native.Stats()
    hw._native.check(hw._native.lib().sacb_get_stats(h, ctypes.byref(st)))
    return st.n_tiles


# name, agents, wide: C1 x 12 (128 x 128 stream tiles, mixed stages split); C2 x 45 (odd count); C2 x 128, the benchmarked population:
# 128 x 256 tiles, light column-sum builds, and arenas more than 2^31 / 2^32 bytes past agent 0's (64-bit agent offsets)
STREAM_POPULATIONS = [("c1_bipedal_m1", 12, False), ("c2_humanoid_m2", 45, False), ("c2_humanoid_m2", 128, True)]


@pytest.mark.parametrize("name,n,wide", STREAM_POPULATIONS)
def test_population_stream_program_equals_single_agents(hw, monkeypatch, name, n, wide):
    """A population whose stages outnumber the SMs takes the throughput form of the program (stream tiles, mixed stages split) -- and
    must still equal the same agents run one by one on the latency form, bitwise: every agent's losses at both steps (step 1 derives
    the weight shadows, step 2 reads the resident ones), and the whole state (nets, targets, Adam moments and steps, alpha) of agents
    0, 1, the last, and the first ones past 2^31 / 2^32 bytes.  The single agents are built one at a time.
    wide: the default program uses 128 x 256 tiles -- a build with SACB_STREAM_N256_MIN=0 (read at each program build) has more
    tiles -- and that build equals the default one bit for bit."""
    from tests.util import population_state, sac_state, selected_agents
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    monkeypatch.delenv("SACB_STREAM_N256_MIN", raising=False)
    case = cases.UPDATE_CASES[name]
    hw.use_networks("model1" if case["n_hidden"] == 2 else "model2")
    obs, act, hid, B = case["obs"], case["act"], case["hidden"], 256
    seeds = list(range(100, 100 + n))
    rng = np.random.RandomState(2)
    data = [O.make_batch(obs, act, 400, seed=900 + i) for i in range(n)]
    idx = [np.stack([rng.permutation(400)[:B] for _ in seeds]).astype(np.int64) for _ in range(2)]
    eps = [(rng.standard_normal((n, B, act)).astype(np.float32), rng.standard_normal((n, B, act)).astype(np.float32)) for _ in range(2)]

    def run_population():
        pop = hw.PopulationSAC(n, obs, act, hidden_dim=hid, device="cuda", seeds=seeds, capacity=512, max_batch=B, seed=7)
        for i, b in enumerate(data):
            pop.push_many(i, b["s"], b["a"], b["r"], b["s2"], b["d"])
        losses = [pop.update_parameters(B, idx=idx[k], eps=eps[k]) for k in range(2)]
        return pop, losses

    pop, losses = run_population()
    sel = selected_agents(pop, require_far=wide)
    states = {i: population_state(pop, i) for i in sel}
    n_tiles = _n_tiles(hw, pop._h)
    del pop
    gc.collect()
    if wide:
        with monkeypatch.context() as mp:
            mp.setenv("SACB_STREAM_N256_MIN", "0")
            narrow, narrow_losses = run_population()
        assert _n_tiles(hw, narrow._h) > n_tiles, (_n_tiles(hw, narrow._h), n_tiles)
        assert narrow_losses == losses
        for i in sel:
            _equal_states(population_state(narrow, i), states[i], f"128-wide tiles, agent {i}")
        del narrow
        gc.collect()
    for i, sd in enumerate(seeds):
        torch.manual_seed(sd)
        ag = hw.SAC(obs, act, hidden_dim=hid, device="cuda", capacity=512, max_batch=B, seed=7)
        ag.replay_buffer.push_many(data[i]["s"], data[i]["a"], data[i]["r"], data[i]["s2"], data[i]["d"])
        for k in range(2):
            ref = ag.update_parameters(B, idx=idx[k][i], eps=(eps[k][0][i], eps[k][1][i]))
            assert losses[k][i] == ref, (k, i, losses[k][i], ref)
        if i in states:
            _equal_states(states[i], sac_state(ag), f"agent {i}")
        del ag
        gc.collect()      # a SAC and its optimizer views reference each other: its handle (device arena) is freed by the collector
    hw.use_networks("model1")
