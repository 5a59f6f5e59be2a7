"""HBM-resident replay buffers behind the reference's replay_buffer.py API.

ReplayBuffer (reference :5-22) and PrioritizedReplayBuffer (:25-90) keep their constructor arguments,
`push` / `sample` / `update_priorities` / `__len__` and the `.buffer` attribute.  Transitions live in a
device ring owned by a `sacb` handle (the SAC agent's when the buffer belongs to one, otherwise a
private one created at the first push, when the observation / action widths become known).
"""
import ctypes
import math
import random
from collections import deque

import numpy as np

from . import _native as N


def _range_sample(n, k):
    """`random.sample(range(n), k)` -- the same picks AND the same consumption of the global `random` stream (so it stays
    interchangeable with the reference's `random.sample(deque, k)`, replay_buffer.py:15, SURVEY H7) -- 5x faster at k = 256.

    CPython's set path (`n > setsize`) draws `randbelow(n)` until the value is new; `randbelow` takes one 32-bit Mersenne
    Twister word per attempt (`getrandbits(n.bit_length())` = word >> (32 - bits), retried while >= n).  So the sample is
    "the first k distinct values < n" of the word stream.  `getrandbits(32 * m)` yields the next m words at once (least
    significant word first); each round draws exactly as many words as picks are still missing -- the minimum the sequential
    loop would also consume -- so the stream never runs ahead.  Small populations (pool path) defer to `random.sample`."""
    if not 0 <= k <= n:
        raise ValueError("Sample larger than population or is negative")
    setsize = 21
    if k > 5:
        setsize += 4 ** math.ceil(math.log(k * 3, 4))
    bits = n.bit_length()
    if n <= setsize or bits > 32 or k == 0:
        return np.asarray(random.sample(range(n), k), np.int64)
    shift, getrandbits = 32 - bits, random.getrandbits
    picks = np.empty(k, np.int64)
    p_picks, first_distinct = N.ptr(picks, ctypes.c_int64), N.lib().sacb_host_first_distinct
    have = 0
    while have < k:      # the filter / first-occurrence rule runs in the library (host code): a numpy formulation costs 2x the time
        need = k - have
        have = first_distinct(getrandbits(32 * need).to_bytes(4 * need, "little"), need, n, shift, p_picks, have, k)
        if have < 0:
            raise RuntimeError("sacb_host_first_distinct: bad argument")
    return picks


def _as_row_parts(state, action, reward, next_state, done):
    s = N.f32(state).ravel()
    a = N.f32(action).ravel()
    s2 = N.f32(next_state).ravel()
    return s, a, np.float32(reward), s2, np.float32(bool(done))


def _transition_arrays(cfg, n):
    """Host arrays (s, a, r, s2, d) for n transitions of a handle with config `cfg`."""
    o, k = cfg.obs_dim, cfg.act_dim
    return (np.empty((n, o), np.float32), np.empty((n, k), np.float32), np.empty(n, np.float32),
            np.empty((n, o), np.float32), np.empty(n, np.float32))


# ---- the prioritized buffer of one agent of a handle: PrioritizedReplayBuffer (agent 0) and PopulationSAC(replay="per") ----------
# `owner` is anything that holds a library handle `_h` and its config `_cfg`.
def _per_priorities(owner, agent):
    """Host copy of the agent's float32[capacity] priority table (zeros for never-written slots)."""
    out = np.zeros(int(owner._cfg.capacity), np.float32)
    N.check(N.lib().sacb_per_get_priorities(owner._h, agent, N.ptr(out), out.size))
    return out


def _per_set_priorities(owner, agent, priorities, p_alpha=None):
    """Overwrite the first len(priorities) entries of the agent's table (p_alpha: its p**alpha table, else computed on the device)."""
    p = N.f32(priorities).ravel()
    pa = None if p_alpha is None else N.f32(p_alpha).ravel()
    if pa is not None and pa.size != p.size:      # the library copies p.size entries of each
        raise ValueError("p_alpha must have one entry per priority")
    N.check(N.lib().sacb_per_set_priorities(owner._h, agent, N.ptr(p), N.ptr(pa), p.size))


def _per_sample(owner, agent, batch_size, u=None):
    """The agent's (s, a, r, s2, d, idx, weights) of min(batch_size, len) rows; `u` = that many uniforms."""
    n = min(batch_size, int(N.lib().sacb_len(owner._h, agent)))                # replay_buffer.py:50
    if n > int(owner._cfg.max_batch):     # one call normalises the IS weights by the batch maximum on the device: no piecewise form
        raise ValueError(f"prioritized sample of {n} rows exceeds the handle's max_batch={int(owner._cfg.max_batch)} "
                         "(standalone buffers: 1024; a buffer of a SAC or PopulationSAC: its max_batch)")
    if u is None:
        u = np.random.random_sample(n)       # the draw np.random.choice(len, n, p=probs) makes (mtrand.pyx::choice)
    u = np.ascontiguousarray(u, np.float64)
    rows = _transition_arrays(owner._cfg, n)
    idx, w = np.empty(n, np.int64), np.empty(n, np.float32)
    N.check(N.lib().sacb_per_sample(owner._h, agent, N.ptr(u, ctypes.c_double), batch_size, N.ptr(idx, ctypes.c_int64), N.ptr(w),
                                    *map(N.ptr, rows)))
    return (*rows, idx, w)


def _per_update_priorities(owner, agent, indices, priorities):
    """The agent's update_priorities: float32 priorities are stored + 1e-6 in float32, float64 ones + 1e-6 in float64."""
    idx = np.ascontiguousarray(np.asarray(indices), np.int64).ravel()
    if hasattr(priorities, "detach"):
        priorities = priorities.detach().cpu().numpy()
    pr = np.asarray(priorities)
    if pr.dtype == np.float32:
        pr = np.ascontiguousarray(pr.ravel())
        N.check(N.lib().sacb_per_update(owner._h, agent, N.ptr(idx, ctypes.c_int64), N.ptr(pr), idx.size))
    else:   # priority.item() + 1e-6 in float64, then the float32 store (replay_buffer.py:87)
        final = (pr.astype(np.float64).ravel() + 1e-6).astype(np.float32)
        N.check(N.lib().sacb_per_update_final(owner._h, agent, N.ptr(idx, ctypes.c_int64), N.ptr(final), idx.size))


def _per_stats(owner, agent):
    st = N.PerStats()
    N.check(N.lib().sacb_per_get_stats(owner._h, agent, ctypes.byref(st)))
    return st


def _per_set_frame(owner, agent, v):
    """The agent's frame counter (beta schedule, replay_buffer.py:53): starts at 1, +1 per sample."""
    N.check(N.lib().sacb_per_set_frame(owner._h, agent, int(v)))


class _DeviceBuffer:
    _KIND = N.REPLAY_UNIFORM

    def __init__(self, capacity):
        self.capacity = int(capacity)
        self._h = None          # sacb handle
        self._owner = None      # SAC agent owning the handle (None: private handle)
        self._cfg = None
        self._pending = []      # packed rows not yet on the device
        self._row_floats = None

    # ---- handle plumbing -------------------------------------------------------------------------------
    def _bind(self, owner):
        self._owner, self._h, self._cfg = owner, owner._h, owner._cfg

    def _extra_config(self, cfg):
        pass

    def _ensure_handle(self, obs_dim, act_dim):
        if self._h is not None:
            return
        cfg = N.default_config()
        cfg.obs_dim, cfg.act_dim, cfg.hidden_dim, cfg.n_hidden = obs_dim, act_dim, 8, 2
        cfg.capacity, cfg.replay_kind, cfg.max_batch = self.capacity, self._KIND, 1024
        self._extra_config(cfg)
        self._cfg = cfg
        self._h = N.create(cfg)

    def __del__(self):
        if getattr(self, "_owner", None) is None and getattr(self, "_h", None) is not None:
            try:
                N.lib().sacb_destroy(self._h)
            except Exception:
                pass

    # ---- push ---------------------------------------------------------------------------------------------
    def push(self, state, action, reward, next_state, done):
        s, a, r, s2, d = _as_row_parts(state, action, reward, next_state, done)
        self._ensure_handle(s.size, a.size)
        if self._row_floats is None:
            self._row_floats = int(N.lib().sacb_row_floats(self._h))
        row = np.zeros(self._row_floats, np.float32)
        o, k = self._cfg.obs_dim, self._cfg.act_dim
        row[:o], row[o:2 * o], row[2 * o:2 * o + k], row[2 * o + k], row[2 * o + k + 1] = s, s2, a, r, d
        self._pending.append(row)
        if len(self._pending) >= 256:
            self._flush()

    def push_many(self, states, actions, rewards, next_states, dones):
        """Bulk push of n transitions (extension; same result as n push() calls)."""
        s, a, s2 = N.f32(states), N.f32(actions), N.f32(next_states)
        r, d = N.f32(rewards).ravel(), N.f32(dones).ravel()
        self._ensure_handle(s.shape[1], a.shape[1])
        self._flush()
        N.check(N.lib().sacb_push(self._h, 0, N.ptr(s), N.ptr(a), N.ptr(r), N.ptr(s2), N.ptr(d), s.shape[0]))

    def _flush(self):
        if self._pending:
            rows = self._pending[0][None, :] if len(self._pending) == 1 else np.ascontiguousarray(np.stack(self._pending))
            self._pending = []
            N.check(N.lib().sacb_push_rows(self._h, 0, N.ptr(rows), rows.shape[0]))

    def __len__(self):
        if self._h is None:
            return 0
        return min(self.capacity, int(N.lib().sacb_len(self._h, 0)) + len(self._pending))

    # ---- host view of the stored transitions (checkpoints read / write `.buffer`, sac_imp.py:199,230) ---------
    def _read(self, idx):
        self._flush()
        idx = np.ascontiguousarray(idx, np.int64)
        rows = _transition_arrays(self._cfg, idx.size)
        N.check(N.lib().sacb_read_transitions(self._h, 0, N.ptr(idx, ctypes.c_int64), idx.size, *map(N.ptr, rows)))
        return rows

    def _materialise(self):
        n = len(self)
        if n == 0:
            return []
        s, a, r, s2, d = self._read(np.arange(n))
        return [(s[i], a[i], float(r[i]), s2[i], bool(d[i])) for i in range(n)]

    def _load(self, transitions):
        if self._h is not None:
            self._pending = []
            N.check(N.lib().sacb_clear_replay(self._h, 0))
        for t in transitions:
            self.push(*t)
        self._flush()


class ReplayBuffer(_DeviceBuffer):
    """replay_buffer.py:5-22: FIFO of capacity 1e6 (deque(maxlen)), uniform sampling WITHOUT replacement."""

    def __init__(self, capacity=1000000):
        super().__init__(capacity)

    @property
    def buffer(self):
        return deque(self._materialise(), maxlen=self.capacity)

    @buffer.setter
    def buffer(self, transitions):
        self._load(list(transitions))

    def _draw(self, batch_size):
        # random.sample(deque, k) and random.sample(range(n), k) pick the same positions and consume the
        # global `random` stream identically (SURVEY H7), so the host draw costs no parity
        return _range_sample(len(self), batch_size)

    def sample(self, batch_size):
        idx = self._draw(batch_size)        # ValueError("Sample larger than population...") like the reference
        self._flush()
        rows = _transition_arrays(self._cfg, idx.size)
        # any size up to len(buffer), like the reference: the library gathers through its staging area in pieces (replay.cu: gather_to_host)
        N.check(N.lib().sacb_sample_uniform(self._h, 0, N.ptr(idx, ctypes.c_int64), idx.size, *map(N.ptr, rows)))
        return rows


class PrioritizedReplayBuffer(_DeviceBuffer):
    """replay_buffer.py:25-90: proportional prioritisation, O(N) inverse-CDF sampling WITH replacement.
    Sampled indices and updated priorities are bit-identical to the reference given the same uniforms."""

    _KIND = N.REPLAY_PER

    def __init__(self, capacity, alpha=0.6, beta_start=0.4, beta_frames=100000):
        super().__init__(capacity)
        self.alpha, self.beta_start, self.beta_frames = alpha, beta_start, beta_frames

    def _extra_config(self, cfg):
        cfg.per_alpha, cfg.per_beta_start, cfg.per_beta_frames = self.alpha, self.beta_start, self.beta_frames

    def _stats(self):
        return _per_stats(self, 0)

    @property
    def frame(self):
        return 1 if self._h is None else int(self._stats().frame)

    @frame.setter
    def frame(self, v):
        _per_set_frame(self, 0, v)

    @property
    def pos(self):
        self._flush()
        return 0 if self._h is None else int(self._stats().pos)

    @property
    def priorities(self):
        """Host copy of the float32[capacity] priority table (zeros for never-written slots)."""
        if self._h is None:
            return np.zeros(self.capacity, np.float32)
        self._flush()
        return _per_priorities(self, 0)

    def set_priorities(self, priorities, p_alpha=None):
        """Overwrite the table (tests: inject numpy's own p**alpha, whose float32 pow is CPU-ISA dependent)."""
        self._flush()
        _per_set_priorities(self, 0, priorities, p_alpha)

    @property
    def buffer(self):
        return self._materialise()

    @buffer.setter
    def buffer(self, transitions):
        self._load(list(transitions))

    def sample(self, batch_size, u=None):
        self._flush()
        return _per_sample(self, 0, batch_size, u)

    def update_priorities(self, indices, priorities):
        self._flush()
        _per_update_priorities(self, 0, indices, priorities)
