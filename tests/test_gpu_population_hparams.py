"""Population-based training on one handle: per-agent hyperparameters, the on-device exploit copy and member checkpoints.

1. A population whose agents all have their own lr, gamma, tau, alpha and target entropy equals the same agents run one by one as
   plain SACs built with those values, bit for bit (latency and throughput forms of the program, fixed and tuned temperature).
2. Hyperparameters changed between two updates act like the same change on single agents, and build no new program.
3. exploit(dst, src): every dst becomes its src, bit for bit, and stays so through an update on the same rows and noise; other agents
   and every replay ring are untouched; malformed index lists raise ValueError.
4. A member's checkpoint resumes as a plain SAC (SAC.load_checkpoint), and a SAC checkpoint resumes as a member: the next update of
   both sides is the same, bit for bit."""
import ctypes
import gc

import numpy as np
import pytest
import torch

from oracle import sac_oracle_np as O
from tests.golden import cases
from tests.util import population_state, sac_state, selected_agents

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hw():
    import humanoid_walking_with_sac_b200 as hw
    yield hw
    hw.use_networks("model1")


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


def hparams_of(n, act):
    """Distinct values for every agent."""
    i = np.arange(n)
    return {"lr": list(3e-4 * (1 + 0.15 * i)), "gamma": list(0.99 - 0.002 * i), "tau": list(0.005 + 0.001 * i),
            "alpha": list(0.2 + 0.01 * i), "target_entropy": list(-float(act) + 0.25 * i)}


def set_target_entropy(hw, h, value):
    N = hw._native
    hp = N.Hparams()
    N.check(N.lib().sacb_get_hparams(h, 0, ctypes.byref(hp)))
    hp.target_entropy = value
    N.check(N.lib().sacb_set_hparams(h, 0, ctypes.byref(hp)))


def single_hparams(hw, h):
    hp = hw._native.Hparams()
    hw._native.check(hw._native.lib().sacb_get_hparams(h, 0, ctypes.byref(hp)))
    return {k: getattr(hp, k) for k in ("lr", "gamma", "tau", "target_entropy")}


def n_programs(hw, h):
    st = hw._native.Stats()
    hw._native.check(hw._native.lib().sacb_get_stats(h, ctypes.byref(st)))
    return st.n_programs


class Setup:
    """n agents of case `name` (seeds 100 + i), `rows` own transitions each, the update inputs of `steps` steps."""

    def __init__(self, hw, name, n, steps, rows=None, B=None):
        self.case = case = cases.UPDATE_CASES[name]
        hw.use_networks("model1" if case["n_hidden"] == 2 else "model2")
        self.hw, self.n = hw, n
        self.obs, self.act, self.hid = case["obs"], case["act"], case["hidden"]
        self.B = B or (24 if name.startswith("tiny") else 256)
        self.rows = rows or (40 if name.startswith("tiny") else 400)
        self.seeds = list(range(100, 100 + n))
        rng = np.random.RandomState(2)
        self.data = [O.make_batch(self.obs, self.act, self.rows, seed=900 + i) for i in range(n)]
        self.idx = [np.stack([rng.permutation(self.rows)[:self.B] for _ in range(n)]).astype(np.int64) for _ in range(steps)]
        self.eps = [(rng.standard_normal((n, self.B, self.act)).astype(np.float32),
                     rng.standard_normal((n, self.B, self.act)).astype(np.float32)) for _ in range(steps)]

    def population(self, hp, auto=True):
        pop = self.hw.PopulationSAC(self.n, self.obs, self.act, hidden_dim=self.hid, device="cuda", seeds=self.seeds, capacity=1024,
                                    max_batch=self.B, seed=7, automatic_entropy_tuning=auto, **hp)
        for i, b in enumerate(self.data):
            pop.push_many(i, b["s"], b["a"], b["r"], b["s2"], b["d"])
        return pop

    def step(self, pop, k):
        return pop.update_parameters(self.B, idx=self.idx[k], eps=self.eps[k])

    def single(self, i, hp, auto=True, seed=None):
        torch.manual_seed(self.seeds[i] if seed is None else seed)
        ag = self.hw.SAC(self.obs, self.act, hidden_dim=self.hid, gamma=hp["gamma"], tau=hp["tau"], lr=hp["lr"], alpha=hp["alpha"],
                         automatic_entropy_tuning=auto, device="cuda", capacity=1024, max_batch=self.B, seed=7)
        set_target_entropy(self.hw, ag._h, hp["target_entropy"])
        b = self.data[i]
        ag.replay_buffer.push_many(b["s"], b["a"], b["r"], b["s2"], b["d"])
        return ag

    def single_step(self, ag, i, k):
        return ag.update_parameters(self.B, idx=self.idx[k][i], eps=(self.eps[k][0][i], self.eps[k][1][i]))


def agent_hp(hp, i):
    return {k: v[i] for k, v in hp.items()}


# ---- 1. heterogeneous population == single agents ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n,auto", [("tiny_m2", 3, True), ("tiny_m2", 3, False), ("c1_bipedal_m1", 12, True), ("c2_humanoid_m2", 45, True)])
def test_heterogeneous_population_equals_single_agents(hw, monkeypatch, name, n, auto):
    """Every agent its own lr, gamma, tau, alpha and target entropy: two updates (the first derives the weight shadows, the second
    reads the resident ones) equal single SACs built with the same values, bitwise -- every agent's losses, and the whole state (nets,
    targets, Adam moments and steps, alpha) and hyperparameters of agents 0, 1 and the last.  tiny_m2 x 3 runs the latency form,
    C1 x 12 and C2 x 45 the throughput (stream) form; auto=False keeps each agent's alpha fixed."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    S = Setup(hw, name, n, steps=2)
    hp = hparams_of(n, S.act)
    pop = S.population(hp, auto)
    for i in range(n):
        got = pop.hyperparameters(i)
        for k, v in agent_hp(hp, i).items():
            assert got[k] == np.float32(v), (i, k, got[k], v)
    losses = [S.step(pop, k) for k in range(2)]
    sel = selected_agents(pop)
    states = {i: population_state(pop, i) for i in sel}
    del pop
    gc.collect()
    for i in range(n):
        ag = S.single(i, agent_hp(hp, i), auto)
        for k in range(2):
            ref = S.single_step(ag, i, k)
            assert losses[k][i] == ref, (k, i, losses[k][i], ref)
        if i in states:
            _equal_states(states[i], sac_state(ag), f"agent {i}")
        del ag
        gc.collect()


# ---- 2. explore between two updates -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n", [("tiny_m2", 3), ("c1_bipedal_m1", 12)])
def test_hyperparameters_changed_mid_run(hw, monkeypatch, name, n):
    """set_hyperparameters (lr included, at step counts 2) between the second and the third update equals single agents changed at the
    same point, bitwise; the third update builds no program (the second already runs the resident-shadow program)."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    S = Setup(hw, name, n, steps=3)
    hp = hparams_of(n, S.act)
    new = {k: v[::-1] for k, v in hparams_of(n, S.act).items()}
    new["lr"] = [x * 0.5 for x in new["lr"]]
    pop = S.population(hp)
    losses = [S.step(pop, k) for k in range(2)]
    built = n_programs(hw, pop._h)
    for i in range(n):
        pop.set_hyperparameters(i, **agent_hp(new, i))
        assert pop.hyperparameters(i) == {k: float(np.float32(v)) for k, v in agent_hp(new, i).items()}
    losses.append(S.step(pop, 2))
    assert n_programs(hw, pop._h) == built
    sel = selected_agents(pop)
    before = pop.hyperparameters(0)      # alpha is the tuned one by now
    pop.set_hyperparameters(0, gamma=0.5)      # only the given key changes
    assert pop.hyperparameters(0) == {**before, "gamma": 0.5}
    states = {i: population_state(pop, i) for i in sel}
    del pop
    gc.collect()
    for i in sel:
        ag = S.single(i, agent_hp(hp, i))
        for k in range(3):
            if k == 2:
                h = agent_hp(new, i)
                N = hw._native
                N.check(N.lib().sacb_set_hparams(ag._h, 0, ctypes.byref(N.Hparams(h["lr"], h["gamma"], h["tau"], h["target_entropy"]))))
                sc = ag._scalars()
                sc.alpha = h["alpha"]
                ag._set_scalars(sc)
            ref = S.single_step(ag, i, k)
            assert losses[k][i] == ref, (k, i, losses[k][i], ref)
        _equal_states(states[i], sac_state(ag), f"agent {i}")
        del ag
        gc.collect()


def test_bad_hyperparameters_raise(hw):
    S = Setup(hw, "tiny_m2", 2, steps=1)
    pop = S.population({})
    before = pop.hyperparameters(1)
    for kw in ({"lr": 0.0}, {"lr": float("inf")}, {"gamma": 1.5}, {"tau": -0.1}, {"target_entropy": float("nan")}, {"alpha": -1.0},
               {"beta": 0.3}):
        with pytest.raises(ValueError):
            pop.set_hyperparameters(1, **kw)
    N = hw._native
    with pytest.raises(ValueError):      # the library refuses the same values on its own
        N.check(N.lib().sacb_set_hparams(pop._h, 1, ctypes.byref(N.Hparams(1e-3, 1.5, 0.005, -1.0))))
    assert pop.hyperparameters(1) == before
    with pytest.raises(ValueError):
        pop.set_hyperparameters(2, lr=1e-3)
    with pytest.raises(ValueError):
        S.population({"gamma": [0.9, 0.99, 0.95]})      # one value per agent


# ---- 3. exploit ------------------------------------------------------------------------------------------------------------------
def _ring(hw, pop, i):
    N = hw._native
    n = pop.buffer_len(i)
    idx = np.arange(n, dtype=np.int64)
    s, s2 = (np.empty((n, pop._cfg.obs_dim), np.float32) for _ in range(2))
    a = np.empty((n, pop._cfg.act_dim), np.float32)
    r, d = np.empty(n, np.float32), np.empty(n, np.float32)
    N.check(N.lib().sacb_read_transitions(pop._h, i, N.ptr(idx, ctypes.c_int64), n, N.ptr(s), N.ptr(a), N.ptr(r), N.ptr(s2), N.ptr(d)))
    return n, s, a, r, s2, d


@pytest.mark.parametrize("name,n,dst,src", [("tiny_m2", 5, [3, 0], [1, 4]), ("c1_bipedal_m1", 12, [11, 2, 5], [0, 7, 7])])
def test_exploit_copies_learner_state(hw, monkeypatch, name, n, dst, src):
    """After two updates, exploit(dst, src): every dst equals its src bitwise (state and hyperparameters), other agents are untouched,
    rings keep their own rows.  Then one update in which each dst gets its src's rows (a block every ring holds alike) and noise:
    dst and src stay equal, losses included."""
    monkeypatch.delenv("SACB_NO_STREAM", raising=False)
    S = Setup(hw, name, n, steps=3)
    shared = O.make_batch(S.obs, S.act, S.rows, seed=777)      # rows [rows, 2 rows) of every ring
    hp = hparams_of(n, S.act)
    pop = S.population(hp)
    for i in range(n):
        pop.push_many(i, shared["s"], shared["a"], shared["r"], shared["s2"], shared["d"])
    for k in range(2):
        S.step(pop, k)
    before = {i: population_state(pop, i) for i in range(n)}
    rings = {i: _ring(hw, pop, i) for i in range(n)}
    pop.exploit(dst, src)
    for i in range(n):
        if i in dst:
            j = src[dst.index(i)]
            _equal_states(population_state(pop, i), before[j], f"dst {i} <- {j}")
            assert pop.hyperparameters(i) == pop.hyperparameters(j)
        else:
            _equal_states(population_state(pop, i), before[i], f"untouched {i}")
        got = _ring(hw, pop, i)
        assert got[0] == rings[i][0] == 2 * S.rows
        for x, y in zip(got[1:], rings[i][1:]):
            np.testing.assert_array_equal(x, y, err_msg=f"ring {i}")
    idx = S.rows + np.stack([np.random.RandomState(40 + i).permutation(S.rows)[:S.B] for i in range(n)]).astype(np.int64)
    e_next, e_cur = S.eps[2][0].copy(), S.eps[2][1].copy()
    for d, s in zip(dst, src):
        idx[d], e_next[d], e_cur[d] = idx[s], e_next[s], e_cur[s]
    losses = pop.update_parameters(S.B, idx=idx, eps=(e_next, e_cur))
    for d, s in zip(dst, src):
        assert losses[d] == losses[s], (d, s, losses[d], losses[s])
        _equal_states(population_state(pop, d), population_state(pop, s), f"after the update, dst {d} <- {s}")
    for bad_dst, bad_src in (([0], [0]), ([1, 1], [2, 3]), ([1, 2], [2, 3]), ([n], [0]), ([0], [-1]), ([0, 1], [2])):
        with pytest.raises(ValueError):
            pop.exploit(bad_dst, bad_src)
    pop.exploit([], [])


# ---- 4. member checkpoints --------------------------------------------------------------------------------------------------------
def test_member_checkpoint_round_trips_through_sac(hw, tmp_path):
    """Member 1 -> agent_checkpoint -> file -> SAC.load_checkpoint: the SAC's next update equals the member's, bitwise (the SAC is
    built with the member's gamma and tau and given its target entropy).  SAC.save_checkpoint -> load_agent_checkpoint(2): member 2
    takes the SAC's state and learning rate, and the next updates agree bitwise as well."""
    S = Setup(hw, "tiny_m2", 3, steps=3)
    hp = hparams_of(3, S.act)
    pop = S.population(hp)
    for k in range(2):
        S.step(pop, k)
    ck = pop.agent_checkpoint(1)
    assert set(ck) == {"policy_state_dict", "q1_state_dict", "q2_state_dict", "q1_target_state_dict", "q2_target_state_dict",
                       "policy_optimizer_state_dict", "q1_optimizer_state_dict", "q2_optimizer_state_dict", "alpha", "log_alpha",
                       "alpha_optimizer_state_dict", "sacb_hyperparameters"}
    torch.save(ck, tmp_path / "member.pt")
    m_hp = {**ck["sacb_hyperparameters"], "alpha": 0.2}
    out = S.single(1, {**m_hp, "lr": 1e-3}, seed=0)      # other weights, another lr: all of it comes from the file
    out.load_checkpoint(str(tmp_path / "member.pt"))
    assert single_hparams(hw, out._h) == ck["sacb_hyperparameters"]
    _equal_states(sac_state(out), population_state(pop, 1), "member 1 as a SAC")

    h2 = pop.hyperparameters(2)
    src = S.single(2, {**h2, "lr": 5e-4}, seed=55)
    for k in range(2):
        S.single_step(src, 2, k)
    src.save_checkpoint(str(tmp_path / "single.pt"), 0, 0, replay_buffer=False)
    pop.load_agent_checkpoint(2, str(tmp_path / "single.pt"))
    assert pop.hyperparameters(2)["lr"] == np.float32(5e-4)
    _equal_states(population_state(pop, 2), sac_state(src), "SAC as member 2")

    losses = S.step(pop, 2)
    assert losses[1] == S.single_step(out, 1, 2)
    assert losses[2] == S.single_step(src, 2, 2)
    _equal_states(population_state(pop, 1), sac_state(out), "member 1 after the next update")
    _equal_states(population_state(pop, 2), sac_state(src), "member 2 after the next update")
