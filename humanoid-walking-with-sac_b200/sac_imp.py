"""Soft Actor-Critic learner behind the reference's sac_imp.SAC API, executed by hand-written sm_100a kernels.

Drop-in surface (reference sac_imp.py): constructor :9-52, select_action :54-72, update_parameters :74-144,
save/load :154-173, save_checkpoint/load_checkpoint :177-233, attributes policy / q1 / q2 / q1_target /
q2_target / *_optimizer / alpha / log_alpha / replay_buffer / gamma / tau / device / target_entropy.

Which networks are used follows the module-level names `QNetwork` / `GaussianPolicy`, exactly like the
reference's `from networks_model1 import ...` (sac_imp.py:4): rebind them to networks_model2's classes to
get the 3x512 variant.  Keyword-only arguments after `device` are extensions (replay kind, math mode...).
"""
import ctypes
import math
import os
import random

import numpy as np
import torch

from . import _native as N
from .networks_model1 import GaussianPolicy, QNetwork
from .replay_buffer import (PrioritizedReplayBuffer, ReplayBuffer, _per_priorities, _per_sample, _per_set_frame, _per_set_priorities,
                            _per_stats, _per_update_priorities)

_NETS = ("policy", "q1", "q2", "q1_target", "q2_target")
_NET_OPTIMIZERS = ((N.NET_POLICY, "policy"), (N.NET_Q1, "q1"), (N.NET_Q2, "q2"))
# torch.optim.Adam's state_dict layout: the param_group entries besides lr / params, and per moment: the arena slot of a network's
# moment, its key in the state, and the scalar-block field of the temperature's (net id None) moment
_ADAM_DEFAULTS = dict(betas=(0.9, 0.999), eps=1e-08, weight_decay=0, amsgrad=False, maximize=False, foreach=None, capturable=False,
                      differentiable=False, fused=None, decoupled_weight_decay=False)
_ADAM_MOMENTS = ((N.SLOT_ADAM_M, "exp_avg", "log_alpha_m"), (N.SLOT_ADAM_V, "exp_avg_sq", "log_alpha_v"))
_STEP_FIELD = {N.NET_POLICY: "step_policy", N.NET_Q1: "step_q1", N.NET_Q2: "step_q2", None: "step_alpha"}


def _adam_group(lr, n_params):
    return dict(lr=lr, **_ADAM_DEFAULTS, params=list(range(n_params)))


def _adam_lr(sd, default=None):
    """Learning rate of a torch.optim.Adam state_dict (`default` if it holds none)."""
    groups = sd.get("param_groups")
    return float(groups[0]["lr"]) if groups and "lr" in groups[0] else default


def _scalar(x):
    """First element of a python number, array or tensor (the device's scalar block holds float32 values)."""
    return float(torch.as_tensor(x).detach().reshape(-1)[0])


def _loss_dict(losses):
    """update_parameters' return value (sac_imp.py:74-144) from a [q1, q2, policy] loss triple."""
    return {"q1_loss": float(losses[0]), "q2_loss": float(losses[1]), "policy_loss": float(losses[2])}


def _config(n_agents, state_dim, action_dim, hidden_dim, n_hidden, policy, gamma, tau, lr, alpha, automatic_entropy_tuning, device, *,
            replay, capacity, max_batch, math, launch, seed, per_alpha, per_beta_start, per_beta_frames, per_weighted_loss, layer_norm=False):
    """The handle's sacb_config from constructor arguments (`policy`: a GaussianPolicy holding the action scale and bias)."""
    cfg = N.default_config()
    cfg.obs_dim, cfg.act_dim, cfg.hidden_dim, cfg.n_hidden = state_dim, action_dim, hidden_dim, n_hidden
    cfg.gamma, cfg.tau, cfg.lr, cfg.alpha0, cfg.auto_entropy = gamma, tau, lr, alpha, int(bool(automatic_entropy_tuning))
    cfg.action_scale, cfg.action_bias = policy.action_scale, policy.action_bias
    cfg.replay_kind = N.REPLAY_PER if replay == "per" else N.REPLAY_UNIFORM
    cfg.capacity, cfg.max_batch, cfg.n_agents, cfg.device = capacity, max_batch, n_agents, torch.device(device).index or 0
    cfg.per_alpha, cfg.per_beta_start, cfg.per_beta_frames = per_alpha, per_beta_start, per_beta_frames
    cfg.per_weighted_loss = int(bool(per_weighted_loss))
    cfg.layer_norm = int(bool(layer_norm))
    cfg.math_mode = {"fp32": N.MATH_FP32, "bf16x3": N.MATH_BF16X3}[math]
    cfg.launch_mode = {"staged": N.LAUNCH_STAGED, "persistent": N.LAUNCH_PERSISTENT}[launch]
    cfg.seed = random.getrandbits(63) if seed is None else int(seed)
    return cfg


def _param_names(module):
    return [(name, tuple(p.shape)) for name, p in module.named_parameters()]


class _Learner:
    """What SAC and PopulationSAC share: a library handle `_h`, and per agent of it the scalar block, the torch.optim.Adam state of
    the four optimizers and the reference's save() / save_checkpoint() layout.  A subclass sets `_cfg` and `_names` (net id -> [(parameter
    name, shape)]) and says where tensors come from: `_tensor`, `_net_state_dicts`, `_load_nets`."""

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None:
            try:
                N.lib().sacb_destroy(h)
            except Exception:
                pass
            self._h = None

    def synchronize(self):
        N.check(N.lib().sacb_synchronize(self._h))

    def _scalars(self, agent=0):
        sc = N.Scalars()
        N.check(N.lib().sacb_get_scalars(self._h, agent, ctypes.byref(sc)))
        return sc

    def _set_scalars(self, sc, agent=0):
        N.check(N.lib().sacb_set_scalars(self._h, agent, ctypes.byref(sc)))

    def _import(self, agent, net_id, slot, t, value):
        host = N.f32(torch.as_tensor(value).detach().cpu().numpy())
        N.check(N.lib().sacb_import_tensor(self._h, agent, net_id, slot, t, N.ptr(host), host.size))

    def _alpha(self, sc, device, alpha_is_float=True):
        """SAC.alpha of the agent whose scalar block is `sc` (a tensor lives on `device`)."""
        if not self._cfg.auto_entropy or sc.n_updates == 0 and alpha_is_float:
            return float(sc.alpha)
        return torch.tensor([sc.alpha], device=device)

    # ---- torch.optim.Adam state of one optimizer of one agent (net_id None: the temperature's) ----------------------------------------
    def _adam_state_dict(self, agent, net_id, sc, lr):
        """state_dict() of the optimizer (scalar block `sc`): like torch, no per-parameter state before the first step."""
        step = getattr(sc, _STEP_FIELD[net_id])
        n = 1 if net_id is None else len(self._names[net_id])
        state = {}
        for t in range(n if step > 0 else 0):
            state[t] = {"step": torch.tensor(float(step))}
            for slot, key, field in _ADAM_MOMENTS:
                state[t][key] = (torch.tensor([getattr(sc, field)]) if net_id is None else
                                 self._tensor(agent, net_id, slot, t, self._names[net_id][t][1]))
        return {"state": state, "param_groups": [_adam_group(lr, n)]}

    def _load_adam_state(self, agent, net_id, sd, sc):
        """Inverse of `_adam_state_dict` into the device and `sc` (the caller stores `sc`).  A parameter without state gets the zero moments
        a fresh torch.optim.Adam starts from; an empty state is step 0."""
        state = sd["state"]
        setattr(sc, _STEP_FIELD[net_id], int(float(state[min(state)]["step"])) if state else 0)
        for slot, key, field in _ADAM_MOMENTS:
            if net_id is None:
                setattr(sc, field, _scalar(state[min(state)][key]) if state else 0.0)
                continue
            for t, (_, shape) in enumerate(self._names[net_id]):
                self._import(agent, net_id, slot, t, state[t][key] if t in state else np.zeros(shape, np.float32))

    # ---- the reference's save() / save_checkpoint() layout of one agent ---------------------------------------------------------------
    def _learner_state(self, agent, device, alpha_is_float=True, lr=None):
        """The learner keys of save() (sac_imp.py:154-162): the five nets and 'alpha'.  Given the learning rate, those of save_checkpoint()
        (:177-201): the optimizers too, and 'log_alpha' with the temperature's optimizer under automatic entropy tuning."""
        sc = self._scalars(agent)
        out = self._net_state_dicts(agent)
        if lr is not None:
            for net_id, name in _NET_OPTIMIZERS:
                out[f"{name}_optimizer_state_dict"] = self._adam_state_dict(agent, net_id, sc, lr)
        out["alpha"] = self._alpha(sc, device, alpha_is_float)
        if lr is not None and self._cfg.auto_entropy:
            out["log_alpha"] = torch.tensor([sc.log_alpha], device=device, requires_grad=True)      # a leaf, like SAC.log_alpha
            out["alpha_optimizer_state_dict"] = self._adam_state_dict(agent, None, sc, lr)
        return out

    def _load_learner(self, agent, checkpoint, optimizers=True):
        """Inverse of `_learner_state`: the nets and alpha; with `optimizers`, each optimizer state and 'log_alpha' the checkpoint holds
        (the temperature's under automatic entropy tuning only).  Returns the learning rate of the last optimizer state that has one."""
        self._load_nets(agent, checkpoint)
        sc, lr = self._scalars(agent), None
        sc.alpha = _scalar(checkpoint["alpha"])
        auto = bool(self._cfg.auto_entropy)
        for net_id, name in (*_NET_OPTIMIZERS, (None, "alpha")) if optimizers else ():
            sd = checkpoint.get(f"{name}_optimizer_state_dict")
            if sd is not None and (net_id is not None or auto):
                self._load_adam_state(agent, net_id, sd, sc)
                lr = _adam_lr(sd, lr)
        if optimizers and auto and "log_alpha" in checkpoint:
            sc.log_alpha = _scalar(checkpoint["log_alpha"])
        self._set_scalars(sc, agent)
        return lr


class ArenaAdam:
    """torch.optim.Adam look-alike over the device arena: the step itself is fused into the update kernels;
    this object only serves `state_dict()` / `load_state_dict()` in the reference checkpoint layout (SURVEY 5)."""

    def __init__(self, owner, net_id, module, lr):
        self._owner, self._net_id = owner, net_id
        self.param_groups = [_adam_group(lr, len(list(module.parameters())) if module is not None else 1)]

    def zero_grad(self, set_to_none=True):
        pass

    def step(self):
        raise RuntimeError("the optimizer step is fused into SAC.update_parameters")

    def state_dict(self):
        return self._owner._adam_state_dict(0, self._net_id, self._owner._scalars(), self.param_groups[0]["lr"])

    def load_state_dict(self, sd):
        sc = self._owner._scalars()
        self._owner._load_adam_state(0, self._net_id, sd, sc)
        self._owner._set_scalars(sc)
        lr = _adam_lr(sd)
        if lr is not None:      # torch.optim.Adam.load_state_dict restores the learning rate of the checkpoint (sac_imp.py:215-218)
            self._owner._set_lr(lr)


class SAC(_Learner):
    """Soft Actor-Critic for continuous actions; one fused device program per update_parameters call."""

    def __init__(self, state_dim, action_dim, hidden_dim=256, gamma=0.99, tau=0.005, lr=3e-4, alpha=0.2,
                 automatic_entropy_tuning=True, device="cuda" if torch.cuda.is_available() else "cpu", *,
                 replay="uniform", capacity=1000000, max_batch=256, math="bf16x3", launch="staged", seed=None,
                 per_alpha=0.6, per_beta_start=0.4, per_beta_frames=100000, per_weighted_loss=False, action_bounds=None, layer_norm=False):
        if not str(device).startswith("cuda"):
            raise RuntimeError("this SAC runs on a B200 only (device='cuda[:i]'); there is no CPU path")
        self.gamma, self.tau, self.device = gamma, tau, device
        self.automatic_entropy_tuning = automatic_entropy_tuning
        self._lr = lr

        # networks: built on the host with the reference's initialisers (same global-RNG consumption order as
        # sac_imp.py:28-36), then uploaded; afterwards every parameter aliases the device arena
        kw = {} if action_bounds is None else {"action_bounds": action_bounds}
        ln = {"layer_norm": True} if layer_norm else {}      # extension, default off (no LayerNorm in the reference): DESIGN.md
        self.layer_norm = bool(layer_norm)
        self.policy = GaussianPolicy(state_dim, action_dim, hidden_dim, **kw, **ln)
        self.q1 = QNetwork(state_dim, action_dim, hidden_dim, **ln)
        self.q2 = QNetwork(state_dim, action_dim, hidden_dim, **ln)
        self.q1_target = QNetwork(state_dim, action_dim, hidden_dim, **ln)
        self.q2_target = QNetwork(state_dim, action_dim, hidden_dim, **ln)
        self.q1_target.load_state_dict(self.q1.state_dict())
        self.q2_target.load_state_dict(self.q2.state_dict())
        n_hidden = getattr(self.q1, "N_HIDDEN", 2)
        if getattr(self.policy, "N_HIDDEN", n_hidden) != n_hidden:
            raise ValueError("QNetwork and GaussianPolicy must come from the same networks_model* variant")

        self._cfg = _config(1, state_dim, action_dim, hidden_dim, n_hidden, self.policy, gamma, tau, lr, alpha, automatic_entropy_tuning, device,
                            replay=replay, capacity=capacity, max_batch=max_batch, math=math, launch=launch, seed=seed,
                            per_alpha=per_alpha, per_beta_start=per_beta_start, per_beta_frames=per_beta_frames,
                            per_weighted_loss=per_weighted_loss, layer_norm=layer_norm)
        self._h = N.create(self._cfg)
        self._arena_base = None
        self._names = {net_id: _param_names(getattr(self, name)) for net_id, name in enumerate(_NETS)}
        for net_id, name in enumerate(_NETS):
            getattr(self, name)._bind(self, net_id)

        self.policy_optimizer = ArenaAdam(self, N.NET_POLICY, self.policy, lr)
        self.q1_optimizer = ArenaAdam(self, N.NET_Q1, self.q1, lr)
        self.q2_optimizer = ArenaAdam(self, N.NET_Q2, self.q2, lr)
        if automatic_entropy_tuning:
            self.target_entropy = -action_dim                                    # sac_imp.py:46
            self.alpha_optimizer = ArenaAdam(self, None, None, lr)

        self.replay_buffer = (PrioritizedReplayBuffer(capacity, per_alpha, per_beta_start, per_beta_frames)
                              if replay == "per" else ReplayBuffer(capacity))
        self.replay_buffer._bind(self)
        self._alpha_is_float = True        # python float until the first update (quirk Q1)
        self._alias_version = None

    def _param_alias(self, net_id, t, shape):
        """Parameter tensor `t` of a network as a VIEW of one tensor spanning the parameter arena: every alias then shares that
        tensor's version counter, and one integer tells whether anything was written through any of them."""
        lib = N.lib()
        if self._arena_base is None:
            lo, hi = None, 0
            for net in range(len(_NETS)):
                for k in range(lib.sacb_num_tensors(self._h, net)):
                    rows, cols, off, dev = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64(), ctypes.c_void_p()
                    N.check(lib.sacb_tensor_info(self._h, net, k, ctypes.byref(rows), ctypes.byref(cols), ctypes.byref(off)))
                    N.check(lib.sacb_tensor_dev(self._h, 0, net, N.SLOT_PARAM, k, ctypes.byref(dev)))
                    lo = dev.value if lo is None else min(lo, dev.value)
                    hi = max(hi, dev.value + 4 * rows.value * cols.value)
            self._arena_base = (lo, torch.as_tensor(N.DevArray(lo, ((hi - lo) // 4,), self), device=f"cuda:{self._cfg.device}"))
        dev = ctypes.c_void_p()
        N.check(lib.sacb_tensor_dev(self._h, 0, net_id, N.SLOT_PARAM, t, ctypes.byref(dev)))
        lo, base = self._arena_base
        first, n = (dev.value - lo) // 4, int(np.prod(shape))
        return base[first:first + n].view(tuple(shape))

    def _publish_alias_writes(self):
        """The GEMMs read bf16 hi/lo shadows that the update's own epilogues keep current.  A write through the torch aliases
        (load_state_dict, `with torch.no_grad(): p.mul_(...)`, ...) bumps the version counter the aliases share (they are views of
        one tensor): the library is then told to re-derive every shadow before the next update.  (`p.data` views have their own
        counter: call invalidate_shadows() after writing through one.)"""
        v = self._arena_base[1]._version
        if v != self._alias_version:
            self._alias_version = v
            N.check(N.lib().sacb_invalidate_shadows(self._h))

    def invalidate_shadows(self):
        N.check(N.lib().sacb_invalidate_shadows(self._h))

    # ---- scalars ---------------------------------------------------------------------------------------------
    def _set_lr(self, lr):
        """The device Adam of all four optimizers shares ONE rate (sac_imp.py:39-49): a new one re-derives its step-size table."""
        N.check(N.lib().sacb_set_lr(self._h, lr))
        self._lr = lr
        for opt in ("policy_optimizer", "q1_optimizer", "q2_optimizer", "alpha_optimizer"):
            if hasattr(self, opt):
                getattr(self, opt).param_groups[0]["lr"] = lr

    def _library_stream(self):
        """The handle's private CUDA stream as a torch stream: torch-side reads / writes of the aliased arena (state_dict,
        load_state_dict, torch.save) are enqueued on it, i.e. ordered against the kernels of the library."""
        if getattr(self, "_ext_stream", None) is None:
            sp = ctypes.c_void_p()
            N.check(N.lib().sacb_get_stream(self._h, ctypes.byref(sp)))
            self._ext_stream = torch.cuda.ExternalStream(sp.value, device=f"cuda:{self._cfg.device}")
        return torch.cuda.stream(self._ext_stream)

    def _tensor(self, agent, net_id, slot, t, shape):
        """A live view of one arena tensor (the state_dicts of this class alias the device memory)."""
        dev = ctypes.c_void_p()
        N.check(N.lib().sacb_tensor_dev(self._h, agent, net_id, slot, t, ctypes.byref(dev)))
        return torch.as_tensor(N.DevArray(dev.value, tuple(shape), self), device=f"cuda:{self._cfg.device}")

    def _net_state_dicts(self, agent):
        return {f"{n}_state_dict": getattr(self, n).state_dict() for n in _NETS}

    def _load_nets(self, agent, checkpoint):
        # the copies into the aliased arena run on the library's own stream (torch's current stream is not ordered against it)
        with self._library_stream():
            for n in _NETS:
                getattr(self, n).load_state_dict(checkpoint[f"{n}_state_dict"])
        self.synchronize()

    @property
    def alpha(self):
        """sac_imp.py:23 / :135: the constructor float until the first tuned update, then exp(log_alpha) (1-element tensor)."""
        return self._alpha(self._scalars(), self.device, self._alpha_is_float)

    @alpha.setter
    def alpha(self, value):
        sc = self._scalars()
        self._alpha_is_float = not torch.is_tensor(value)
        sc.alpha = _scalar(value)
        self._set_scalars(sc)

    @property
    def log_alpha(self):
        # a leaf that requires grad, like the reference's (sac_imp.py:48): a checkpoint written here stays trainable when the
        # reference's load_checkpoint (sac_imp.py:222-223) rebinds `self.log_alpha` to the loaded tensor
        return torch.tensor([self._scalars().log_alpha], device=self.device, requires_grad=True)

    @log_alpha.setter
    def log_alpha(self, value):
        sc = self._scalars()
        sc.log_alpha = _scalar(value)
        self._set_scalars(sc)

    # ---- acting ----------------------------------------------------------------------------------------------
    def select_action(self, state, evaluate=False, *, eps=None):
        """sac_imp.py:54-72: B=1 policy evaluation on the device; `eps` (test hook) replaces the on-device N(0,1) draw."""
        obs = N.f32(state).ravel()
        out = np.empty(self._cfg.act_dim, np.float32)
        e = None if eps is None else N.f32(eps).ravel()
        N.check(N.lib().sacb_select_action(self._h, 0, N.ptr(obs), int(bool(evaluate)), N.ptr(e), N.ptr(out)))
        return out

    # ---- learning --------------------------------------------------------------------------------------------
    def update_parameters(self, batch_size=256, *, eps=None, idx=None, u=None, sync=True):
        """sac_imp.py:74-144.  Draws the minibatch like the reference (`random.sample` positions for the uniform
        buffer, inverse-CDF with `np.random.random_sample` uniforms for the prioritized one), runs the fused update.
        Test hooks: `eps=(eps_next, eps_cur)` [B,act] arrays, `idx` positions, `u` uniforms.  sync=False skips the
        blocking read of the three losses (returns None)."""
        buf = self.replay_buffer
        lib = N.lib()
        self._publish_alias_writes()
        e_next = e_cur = None
        if eps is not None:
            e_next, e_cur = N.f32(eps[0]), N.f32(eps[1])
        losses = np.zeros(3, np.float32)
        flags = 0 if sync else N.NO_LOSS_READBACK
        per = isinstance(buf, PrioritizedReplayBuffer)
        if per:      # host-side draws first: everything behind the flush is then enqueued back to back
            n = min(batch_size, len(buf))
            uu = np.ascontiguousarray(np.random.random_sample(n) if u is None else u, np.float64)
        else:
            ix = buf._draw(batch_size) if idx is None else np.ascontiguousarray(idx, np.int64)
        buf._flush()
        if per:
            N.check(lib.sacb_per_sample(self._h, 0, N.ptr(uu, ctypes.c_double), batch_size, None, None, None, None, None, None, None))
            if self._cfg.per_weighted_loss:      # update_priorities(|q1 - y|): enqueued by the same call, behind the loss copy
                flags |= N.WRITE_BACK_TD
            N.check(lib.sacb_update(self._h, n, None, N.ptr(e_next), N.ptr(e_cur), N.ptr(losses) if sync else None, flags | N.USE_LAST_SAMPLE))
        else:
            N.check(lib.sacb_update(self._h, ix.size, N.ptr(ix, ctypes.c_int64), N.ptr(e_next), N.ptr(e_cur), N.ptr(losses) if sync else None, flags))
        self._alpha_is_float = False
        if not sync:
            return None
        return _loss_dict(losses)

    def learner_steps(self, batch_size=256, k=8, *, sync=True):
        """K learner steps per call, nothing of a step on the host (SURVEY 8f rank 3; trainer.py:190-205 with the updates of K
        environment steps batched): prioritized ring = K x the `learner_step` pipeline, uniform ring = K updates whose positions are
        drawn inside the gather stage (a keyed bijection of range(len): distinct positions, like random.sample); eps on the device;
        ONE read-back of the K loss triples.  Bitwise equal to K single calls.  Returns a list of K dicts (sync=False: None)."""
        self.replay_buffer._flush()
        self._publish_alias_writes()
        losses = np.zeros((k, 3), np.float32)
        N.check(N.lib().sacb_update_steps(self._h, batch_size, k, N.ptr(losses) if sync else None, 0 if sync else N.NO_LOSS_READBACK))
        self._alpha_is_float = False
        if not sync:
            return None
        return [_loss_dict(l) for l in losses]

    def learner_step(self, batch_size=256, *, sync=False):
        """Throughput form of `update_parameters` over the prioritized buffer (per_weighted_loss mode), everything resident
        in HBM: update on the minibatch sampled by the previous call -> priorities <- |q1 - y| -> sample for the next call;
        the write-back and the sample run on a second stream under the rest of the update (`sacb_per_step`).  Device-drawn
        uniforms and eps.  Same values as `update_parameters` with device draws; a transition pushed between two calls
        can first be drawn one call later."""
        buf = self.replay_buffer
        if not isinstance(buf, PrioritizedReplayBuffer):
            raise ValueError("learner_step needs the prioritized replay buffer")
        buf._flush()
        self._publish_alias_writes()
        losses = np.zeros(3, np.float32)
        N.check(N.lib().sacb_per_step(self._h, batch_size, N.ptr(losses) if sync else None, 0 if sync else N.NO_LOSS_READBACK))
        self._alpha_is_float = False
        if not sync:
            return None
        return _loss_dict(losses)

    def update_from_batch(self, batch, eps=None, is_weights=None, export_grads=False, want_td=False):
        """Same step on a caller-supplied minibatch dict(s,a,r,s2,d) (parity tests / benchmarks; no replay involved)."""
        s, a, r, s2, d = (N.f32(batch[k]) for k in ("s", "a", "r", "s2", "d"))
        B = s.shape[0]
        self._publish_alias_writes()
        e_next = e_cur = None
        if eps is not None:
            e_next, e_cur = N.f32(eps[0]), N.f32(eps[1])
        w = None if is_weights is None else N.f32(is_weights)
        losses = np.zeros(3, np.float32)
        td = np.empty(B, np.float32) if want_td else None
        N.check(N.lib().sacb_update_batch(self._h, B, N.ptr(s), N.ptr(a), N.ptr(r), N.ptr(s2), N.ptr(d), N.ptr(w), N.ptr(e_next), N.ptr(e_cur),
                                          N.ptr(losses), N.ptr(td), N.EXPORT_GRADS if export_grads else 0))
        self._alpha_is_float = False
        out = _loss_dict(losses)
        return (out, td) if want_td else out

    def exported_grads(self, net):
        """Gradients of the last update run with export_grads=True, keyed like `named_parameters()`."""
        net_id = {"policy": N.NET_POLICY, "q1": N.NET_Q1, "q2": N.NET_Q2}[net]
        module = getattr(self, net)
        return {name: self._tensor(0, net_id, N.SLOT_GRAD, i, p.shape).cpu().numpy() for i, (name, p) in enumerate(module.named_parameters())}

    def _soft_update_target_networks(self):
        raise RuntimeError("the Polyak update is fused into update_parameters (sac_imp.py:146-152)")

    # ---- persistence (same dictionary keys as the reference) ----------------------------------------------------
    def save(self, path):
        self.synchronize()                  # an update enqueued with sync=False / learner_step may still be running
        with self._library_stream():
            torch.save(self._learner_state(0, self.device, self._alpha_is_float), path)

    def load(self, path):
        checkpoint = torch.load(path, map_location=self.device, weights_only=False)
        self._load_learner(0, checkpoint, optimizers=False)
        self._alpha_is_float = not torch.is_tensor(checkpoint["alpha"])

    def save_checkpoint(self, path, episode, total_steps, replay_buffer=True, *, rng_state=False):
        """sac_imp.py:177-201, same keys.  rng_state=True adds one extra key ('sacb_rng_state': the Philox counters of the
        on-device eps / exploration draws) so that a seeded run resumes its own random stream; the reference ignores it."""
        self.synchronize()
        with self._library_stream():
            checkpoint = {"episode": episode, "total_steps": total_steps, **self._learner_state(0, self.device, self._alpha_is_float, self._lr)}
            if replay_buffer:
                checkpoint["replay_buffer"] = self.replay_buffer.buffer
            if rng_state:
                sc = self._scalars()
                checkpoint["sacb_rng_state"] = {"seed": int(self._cfg.seed), "n_updates": int(sc.n_updates), "act_counter": int(sc.act_counter)}
            # the reference only writes the file inside `if replay_buffer:` (sac_imp.py:198-201); always writing is the fix
            torch.save(checkpoint, path)

    def load_checkpoint(self, path, load_replay_buffer=True):
        checkpoint = torch.load(path, map_location=self.device, weights_only=False)   # pickled deque / numpy inside
        lr = self._load_learner(0, checkpoint)
        self._alpha_is_float = not torch.is_tensor(checkpoint["alpha"])
        if lr is not None:
            self._set_lr(lr)
        if load_replay_buffer and "replay_buffer" in checkpoint:
            self.replay_buffer.buffer = checkpoint["replay_buffer"]
        rs = checkpoint.get("sacb_rng_state")
        if rs is not None and int(rs.get("seed", -1)) == int(self._cfg.seed):      # resume this seed's Philox streams where they stopped
            sc = self._scalars()
            sc.n_updates, sc.act_counter = int(rs["n_updates"]), int(rs["act_counter"])
            self._set_scalars(sc)
        return checkpoint.get("episode", 0), checkpoint.get("total_steps", 0)

    # ---- instrumentation ------------------------------------------------------------------------------------------
    def stats(self):
        st = N.Stats()
        N.check(N.lib().sacb_get_stats(self._h, ctypes.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}


class PopulationSAC(_Learner):
    """`n_agents` independent SAC agents (distinct seeds) trained by ONE batched update program per step on one GPU
    (BASELINE.json configs[4]; the per-agent step is sac_imp.py:74-144).  Agent i = exactly what `torch.manual_seed(seeds[i]);
    SAC(state_dim, action_dim, ...)` builds: same initialiser calls in the same order, its own Adam state, temperature, Philox stream
    (stream id = agent index) and its own uniform replay ring of `capacity` transitions in HBM -- the agent index is a grid
    dimension of every stage kernel and the 4th coordinate of the TMA descriptors.  No inter-agent (or inter-GPU) traffic:
    `distributed.partition_agents` assigns global agent ids to ranks.  Minibatch positions are drawn on the device.

    replay="per": every agent gets its own prioritized buffer instead (replay_buffer.py:25-90 each: priority table, max-priority
    rule, frame counter and beta schedule per agent; `capacity` <= 2 096 128 per agent).  One chain of three sampler launches draws
    every agent's minibatch, one launch writes every agent's |TD| priorities back (`per_weighted_loss`, as in `SAC`).  Per-agent
    accessors mirror PrioritizedReplayBuffer: `priorities`, `set_priorities`, `sample`, `update_priorities`, `frame`, `set_frame`.

    Population-based training: `gamma`, `tau`, `lr`, `alpha` and `target_entropy` (default -action_dim, sac_imp.py:46) take one value
    for all agents or one per agent.  They live in each agent's scalar block on the device, so `set_hyperparameters` (explore) never
    rebuilds the update program, and `exploit(dst, src)` copies whole learner states on the device.  `automatic_entropy_tuning` is
    shared by all agents."""

    HPARAMS = ("lr", "gamma", "tau", "target_entropy", "alpha")

    def __init__(self, n_agents, state_dim, action_dim, hidden_dim=256, gamma=0.99, tau=0.005, lr=3e-4, alpha=0.2,
                 automatic_entropy_tuning=True, device="cuda", *, seeds=None, capacity=100000, max_batch=256, math="bf16x3",
                 launch="staged", seed=None, action_bounds=None, target_entropy=None, replay="uniform", per_alpha=0.6, per_beta_start=0.4,
                 per_beta_frames=100000, per_weighted_loss=False):
        if not str(device).startswith("cuda"):
            raise RuntimeError("PopulationSAC runs on a B200 only (device='cuda[:i]'); there is no CPU path")
        if replay not in ("uniform", "per"):
            raise ValueError(f"replay must be 'uniform' or 'per', got {replay!r}")
        self._per = replay == "per"
        self.n_agents, self.device = int(n_agents), device
        self.seeds = list(range(self.n_agents)) if seeds is None else [int(x) for x in seeds]
        if len(self.seeds) != self.n_agents:
            raise ValueError("one seed per agent")
        hp = {k: self._per_agent(k, v) for k, v in (("lr", lr), ("gamma", gamma), ("tau", tau), ("alpha", alpha),
                                                     ("target_entropy", -float(action_dim) if target_entropy is None else target_entropy))}
        for i in range(self.n_agents):
            self._check_hparams({k: v[i] for k, v in hp.items()})
        kw = {} if action_bounds is None else {"action_bounds": action_bounds}
        probe = GaussianPolicy(state_dim, action_dim, hidden_dim, **kw)
        self._cfg = cfg = _config(self.n_agents, state_dim, action_dim, hidden_dim, getattr(probe, "N_HIDDEN", 2), probe,
                                  hp["gamma"][0], hp["tau"][0], hp["lr"][0], hp["alpha"][0], automatic_entropy_tuning, device,
                                  replay=replay, capacity=capacity, max_batch=max_batch, math=math, launch=launch, seed=seed,
                                  per_alpha=per_alpha, per_beta_start=per_beta_start, per_beta_frames=per_beta_frames,
                                  per_weighted_loss=per_weighted_loss)
        self._h = N.create(cfg)
        self._names = {}
        for i, sd in enumerate(self.seeds):
            torch.manual_seed(sd)                      # the construction order of sac_imp.py:28-36 under this agent's seed
            pol = GaussianPolicy(state_dim, action_dim, hidden_dim, **kw)
            q1, q2 = QNetwork(state_dim, action_dim, hidden_dim), QNetwork(state_dim, action_dim, hidden_dim)
            QNetwork(state_dim, action_dim, hidden_dim); QNetwork(state_dim, action_dim, hidden_dim)     # the targets' own (discarded) init draws
            for net_id, mod in ((N.NET_POLICY, pol), (N.NET_Q1, q1), (N.NET_Q2, q2), (N.NET_Q1_TARGET, q1), (N.NET_Q2_TARGET, q2)):
                self._names[net_id] = _param_names(mod)
                for t, p in enumerate(mod.parameters()):
                    self._import(i, net_id, N.SLOT_PARAM, t, p)
        default = (cfg.lr, cfg.gamma, cfg.tau, -float(action_dim), cfg.alpha0)
        for i in range(self.n_agents):
            mine = {k: float(np.float32(hp[k][i])) for k in self.HPARAMS}
            if tuple(mine.values()) != tuple(float(np.float32(x)) for x in default):
                self.set_hyperparameters(i, **mine)

    def __len__(self):
        return self.n_agents

    # ---- replay (per-agent uniform ring, replay_buffer.py:5-22) -------------------------------------------------------
    def push(self, agent, state, action, reward, next_state, done):
        self.push_many(agent, N.f32(state)[None], N.f32(action)[None], [reward], N.f32(next_state)[None], [done])

    def push_many(self, agent, states, actions, rewards, next_states, dones):
        s, a, s2 = N.f32(states), N.f32(actions), N.f32(next_states)
        r, d = N.f32(rewards).ravel(), N.f32(dones).ravel()
        N.check(N.lib().sacb_push(self._h, int(agent), N.ptr(s), N.ptr(a), N.ptr(r), N.ptr(s2), N.ptr(d), s.shape[0]))

    def buffer_len(self, agent):
        return int(N.lib().sacb_len(self._h, int(agent)))

    # ---- per-agent prioritized buffer (replay="per"; PrioritizedReplayBuffer's interface with an agent index) -------------------------
    def _per_agent_index(self, agent):
        if not self._per:
            raise ValueError("this population has uniform replay rings (construct it with replay='per')")
        return self._agent_index(agent)

    def priorities(self, agent):
        """Host copy of agent `agent`'s float32[capacity] priority table (zeros for never-written slots)."""
        return _per_priorities(self, self._per_agent_index(agent))

    def set_priorities(self, agent, priorities, p_alpha=None):
        """Overwrite the first len(priorities) entries of one agent's table (p_alpha: its p**alpha table, else computed on the device)."""
        _per_set_priorities(self, self._per_agent_index(agent), priorities, p_alpha)

    def sample(self, agent, batch_size, u=None):
        """PrioritizedReplayBuffer.sample of one agent: (s, a, r, s2, d, idx, weights); `u` = its min(batch_size, len) uniforms."""
        return _per_sample(self, self._per_agent_index(agent), batch_size, u)

    def update_priorities(self, agent, indices, priorities):
        """PrioritizedReplayBuffer.update_priorities of one agent (float32 priorities are stored + 1e-6 in float32, float64 ones in float64)."""
        _per_update_priorities(self, self._per_agent_index(agent), indices, priorities)

    def frame(self, agent):
        """The agent's frame counter (beta schedule, replay_buffer.py:53): starts at 1, +1 per sample of that agent."""
        return int(_per_stats(self, self._per_agent_index(agent)).frame)

    def set_frame(self, agent, v):
        _per_set_frame(self, self._per_agent_index(agent), v)

    # ---- acting / learning ------------------------------------------------------------------------------------------------
    def select_action(self, states, evaluate=False, *, eps=None):
        """states [n_agents, obs] -> actions [n_agents, act]: agent i acts on row i with its own policy (sac_imp.py:54-72 each)."""
        obs = N.f32(states).reshape(self.n_agents, self._cfg.obs_dim)
        out = np.empty((self.n_agents, self._cfg.act_dim), np.float32)
        e = None if eps is None else N.f32(eps).reshape(self.n_agents, self._cfg.act_dim)
        N.check(N.lib().sacb_select_action_batch(self._h, N.ptr(obs), int(bool(evaluate)), N.ptr(e), N.ptr(out)))
        return out

    def update_parameters(self, batch_size=256, *, idx=None, u=None, eps=None, sync=True):
        """One update of EVERY agent (sac_imp.py:74-144 each) in one program.  idx [n_agents, B] positions / eps = (eps_next,
        eps_cur) [n_agents, B, act] are test hooks; by default both are drawn on the device.  Returns a list of loss dicts.
        replay="per": every agent's minibatch is one prioritized sample of B rows (each agent's buffer must hold at least B transitions),
        drawn for all agents at once; `u` [n_agents, B] replaces the uniforms drawn on the device (idx does not apply).  With
        per_weighted_loss the critic loss is IS-weighted and every agent's priorities of its minibatch become |q1 - y| + 1e-6."""
        lib = N.lib()
        e_next = e_cur = None
        if eps is not None:
            e_next, e_cur = N.f32(eps[0]), N.f32(eps[1])
        if self._per:
            if idx is not None:
                raise ValueError("a prioritized population draws its minibatches with the sampler: pass u, not idx")
            uu = None if u is None else np.ascontiguousarray(u, np.float64).reshape(self.n_agents, batch_size)
            N.check(lib.sacb_per_sample_all(self._h, N.ptr(uu, ctypes.c_double), batch_size, None, None))
            flags = N.NO_LOSS_READBACK | N.USE_LAST_SAMPLE | (N.WRITE_BACK_TD if self._cfg.per_weighted_loss else 0)
            N.check(lib.sacb_update(self._h, batch_size, None, N.ptr(e_next), N.ptr(e_cur), None, flags))
        elif u is not None:
            raise ValueError("u: uniforms of the prioritized sampler (replay='per')")
        elif idx is not None:
            ix = np.ascontiguousarray(idx, np.int64).reshape(self.n_agents, batch_size)
            N.check(lib.sacb_update(self._h, batch_size, N.ptr(ix, ctypes.c_int64), N.ptr(e_next), N.ptr(e_cur), None, N.NO_LOSS_READBACK))
        else:
            N.check(lib.sacb_update(self._h, batch_size, None, N.ptr(e_next), N.ptr(e_cur), None, N.NO_LOSS_READBACK | N.DEVICE_INDICES))
        if not sync:
            return None
        losses = np.zeros((self.n_agents, 3), np.float32)
        N.check(lib.sacb_get_losses_all(self._h, N.ptr(losses)))
        return [_loss_dict(l) for l in losses]

    # ---- per-agent state in the reference's save() layout (sac_imp.py:154-162) ---------------------------------------
    def _tensor(self, agent, net_id, slot, t, shape):
        """A host copy of one arena tensor of `agent`."""
        host = np.empty(shape, np.float32)
        N.check(N.lib().sacb_export_tensor(self._h, agent, net_id, slot, t, N.ptr(host), host.size))
        return torch.from_numpy(host)

    def _net_state_dicts(self, agent):
        out = {}
        for net_id, name in enumerate(_NETS):
            out[f"{name}_state_dict"] = {pname: self._tensor(agent, net_id, N.SLOT_PARAM, t, shape)
                                         for t, (pname, shape) in enumerate(self._names[net_id])}
        return out

    def _load_nets(self, agent, checkpoint):
        for net_id, name in enumerate(_NETS):
            sd = checkpoint[f"{name}_state_dict"]
            for t, (pname, _) in enumerate(self._names[net_id]):
                self._import(agent, net_id, N.SLOT_PARAM, t, sd[pname])

    def agent_state(self, agent):
        return self._learner_state(int(agent), None)

    def load_agent(self, agent, checkpoint):
        """Inverse of `agent_state` (accepts a file written by the reference's or the product's `SAC.save`)."""
        self._load_learner(int(agent), checkpoint, optimizers=False)

    # ---- population-based training: per-agent hyperparameters, exploit, member checkpoints ---------------------------------------------
    def _per_agent(self, name, value):
        if np.ndim(value) == 0:
            return [float(value)] * self.n_agents
        vals = [float(x) for x in value]
        if len(vals) != self.n_agents:
            raise ValueError(f"{name}: one value or one per agent ({self.n_agents}), got {len(vals)}")
        return vals

    @staticmethod
    def _check_hparams(hp):
        """The library refuses the same values (sacb_set_hparams); alpha is checked here because it travels in sacb_set_scalars."""
        if "alpha" in hp and not (math.isfinite(hp["alpha"]) and hp["alpha"] >= 0):
            raise ValueError(f"alpha must be finite and >= 0, got {hp['alpha']}")
        if "lr" in hp and not (math.isfinite(hp["lr"]) and hp["lr"] > 0):
            raise ValueError(f"lr must be finite and > 0, got {hp['lr']}")
        for k in ("gamma", "tau"):
            if k in hp and not 0.0 <= hp[k] <= 1.0:
                raise ValueError(f"{k} must lie in [0, 1], got {hp[k]}")
        if "target_entropy" in hp and not math.isfinite(hp["target_entropy"]):
            raise ValueError(f"target_entropy must be finite, got {hp['target_entropy']}")

    def _agent_index(self, agent):
        i = int(agent)
        if not 0 <= i < self.n_agents:
            raise ValueError(f"agent {agent} out of range [0, {self.n_agents})")
        return i

    def hyperparameters(self, agent):
        """{lr, gamma, tau, target_entropy, alpha} of one agent as the device holds them (float32 values)."""
        i, hp = self._agent_index(agent), N.Hparams()
        N.check(N.lib().sacb_get_hparams(self._h, i, ctypes.byref(hp)))
        return {"lr": hp.lr, "gamma": hp.gamma, "tau": hp.tau, "target_entropy": hp.target_entropy, "alpha": self._scalars(i).alpha}

    def set_hyperparameters(self, agent, **kw):
        """Explore step: change only the given keys of one agent, effective from its next update (no program is rebuilt).  A new lr
        applies to all four optimizers of the agent from their current step counts; a new alpha is the temperature of the next update
        (with automatic entropy tuning, log_alpha keeps its value and the tuned alpha takes over after that update)."""
        i, lib = self._agent_index(agent), N.lib()
        unknown = set(kw) - set(self.HPARAMS)
        if unknown:
            raise ValueError(f"unknown hyperparameters {sorted(unknown)}; known: {self.HPARAMS}")
        kw = {k: float(v) for k, v in kw.items()}
        self._check_hparams(kw)
        if set(kw) - {"alpha"}:
            cur = N.Hparams()
            N.check(lib.sacb_get_hparams(self._h, i, ctypes.byref(cur)))
            for k in ("lr", "gamma", "tau", "target_entropy"):
                if k in kw:
                    setattr(cur, k, kw[k])
            N.check(lib.sacb_set_hparams(self._h, i, ctypes.byref(cur)))
        if "alpha" in kw:
            sc = self._scalars(i)
            sc.alpha = kw["alpha"]
            self._set_scalars(sc, i)

    def exploit(self, dst, src):
        """Exploit step: agent dst[k] takes over the whole learner state of agent src[k] (weights, targets, Adam state, temperature,
        hyperparameters, step counts), copied on the device.  Replay rings -- and with replay="per" the priority tables and frame
        counters -- stay with their agent, and dst[k] keeps drawing its own minibatch positions and noise (the device streams are keyed
        by agent index).  A dst may appear once, and no agent may be both
        a src and a dst of the same call (ValueError)."""
        d = np.ascontiguousarray(np.asarray(dst, np.int64).ravel())
        s = np.ascontiguousarray(np.asarray(src, np.int64).ravel())
        if d.size != s.size:
            raise ValueError("exploit: dst and src must have the same length")
        if d.size and (min(d.min(), s.min()) < 0 or max(d.max(), s.max()) >= self.n_agents):
            raise ValueError(f"exploit: agent index out of range [0, {self.n_agents})")
        d32, s32 = d.astype(np.int32), s.astype(np.int32)
        N.check(N.lib().sacb_copy_agents(self._h, N.ptr(d32, ctypes.c_int32), N.ptr(s32, ctypes.c_int32), int(d.size)))

    def agent_checkpoint(self, agent):
        """One member as a dictionary in the key layout of SAC.save_checkpoint without 'replay_buffer' (torch.save it): the five nets,
        the three optimizer state_dicts, 'alpha', 'log_alpha' and 'alpha_optimizer_state_dict' (with automatic entropy tuning), and the
        extension key 'sacb_hyperparameters' ({lr, gamma, tau, target_entropy}).  SAC.load_checkpoint accepts the file: that is how a
        member leaves the population (SAC keeps its own gamma / tau / target_entropy; pass them to its constructor or sacb_set_hparams)."""
        i = self._agent_index(agent)
        self.synchronize()
        hp = self.hyperparameters(i)
        ck = self._learner_state(i, None, lr=hp["lr"])
        ck["sacb_hyperparameters"] = {k: hp[k] for k in ("lr", "gamma", "tau", "target_entropy")}
        return ck

    def load_agent_checkpoint(self, agent, checkpoint):
        """Inverse of `agent_checkpoint`; also takes a file (or dictionary) written by SAC.save_checkpoint.  Loads the nets, the Adam
        state and step counts, alpha and log_alpha, and the hyperparameters: 'sacb_hyperparameters' when present, otherwise the
        optimizers' learning rate (gamma, tau and target_entropy of the member then stay as they are)."""
        i = self._agent_index(agent)
        if isinstance(checkpoint, (str, bytes, os.PathLike)):
            checkpoint = torch.load(checkpoint, map_location="cpu", weights_only=False)
        lr = self._load_learner(i, checkpoint)
        hp = checkpoint.get("sacb_hyperparameters")
        if hp is None:
            hp = {} if lr is None else {"lr": lr}
        self.set_hyperparameters(i, **hp)
