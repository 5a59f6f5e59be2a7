"""CPU-side checks of the drop-in boundary: the library loads, exports every symbol include/sacb200.h declares,
the Python mirror keeps the reference signatures, and compute entry points fail loudly without a GPU."""
import inspect
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hw():
    import __graft_entry__
    __graft_entry__.build()
    import humanoid_walking_with_sac_b200 as hw
    return hw


def test_every_declared_symbol_is_exported_and_bound(hw):
    header = open(os.path.join(ROOT, "include", "sacb200.h")).read()
    declared = set(re.findall(r"\b(sacb_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 40
    lib = hw._native.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in sacb200.h but not exported"
        assert name in hw._native.SIGNATURES, f"{name} has no ctypes signature"
    assert set(hw._native.SIGNATURES) == declared


def test_config_struct_matches_header(hw):
    import ctypes
    cfg = hw._native.default_config()
    assert ctypes.sizeof(cfg) == 132 or ctypes.sizeof(cfg) % 8 == 0
    assert (cfg.hidden_dim, cfg.n_hidden, cfg.max_batch, cfg.capacity) == (256, 2, 256, 1000000)
    assert abs(cfg.gamma - 0.99) < 1e-7 and abs(cfg.tau - 0.005) < 1e-9 and abs(cfg.lr - 3e-4) < 1e-9 and abs(cfg.alpha0 - 0.2) < 1e-7
    assert abs(cfg.per_alpha - 0.6) < 1e-7 and abs(cfg.per_beta_start - 0.4) < 1e-7 and cfg.per_beta_frames == 100000


def test_enumerators_match_header(hw):
    """every `SACB_<NAME> = <int>` of include/sacb200.h (status codes, modes, net / slot ids, update flags) has the same value in the binding"""
    hdr = open(os.path.join(ROOT, "include", "sacb200.h")).read()
    found = re.findall(r"\bSACB_([A-Z0-9_]+)\s*=\s*(-?\d+)", hdr)
    assert len(found) >= 25
    for name, val in found:
        assert getattr(hw._native, name) == int(val), name


def test_reference_signatures_are_mirrored(hw):
    """Positional parameters of the reference API (sac_imp.py:9-20, :54, :74; replay_buffer.py:7, :26)."""
    sig = inspect.signature(hw.SAC.__init__)
    names = [p.name for p in sig.parameters.values() if p.kind == p.POSITIONAL_OR_KEYWORD]
    assert names == ["self", "state_dim", "action_dim", "hidden_dim", "gamma", "tau", "lr", "alpha", "automatic_entropy_tuning", "device"]
    d = {k: v.default for k, v in sig.parameters.items()}
    assert (d["hidden_dim"], d["gamma"], d["tau"], d["lr"], d["alpha"], d["automatic_entropy_tuning"]) == (256, 0.99, 0.005, 3e-4, 0.2, True)
    assert list(inspect.signature(hw.SAC.select_action).parameters)[:3] == ["self", "state", "evaluate"]
    assert inspect.signature(hw.SAC.update_parameters).parameters["batch_size"].default == 256
    assert inspect.signature(hw.ReplayBuffer.__init__).parameters["capacity"].default == 1000000
    p = inspect.signature(hw.PrioritizedReplayBuffer.__init__).parameters
    assert (p["alpha"].default, p["beta_start"].default, p["beta_frames"].default) == (0.6, 0.4, 100000)
    for cls in (hw.ReplayBuffer, hw.PrioritizedReplayBuffer):
        assert list(inspect.signature(cls.push).parameters) == ["self", "state", "action", "reward", "next_state", "done"]
    for meth in ("save", "load", "save_checkpoint", "load_checkpoint"):
        assert hasattr(hw.SAC, meth)


def test_network_modules_keep_reference_layout(hw):
    q1 = hw.networks_model1.QNetwork(24, 4)
    assert [k for k in q1.state_dict()] == ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias"]
    assert tuple(q1.fc1.weight.shape) == (256, 28) and tuple(q1.fc3.weight.shape) == (1, 256)
    p2 = hw.networks_model2.GaussianPolicy(348, 17, device="cpu")
    assert [k for k in p2.state_dict()] == ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias",
                                            "mean.weight", "mean.bias", "log_std.weight", "log_std.bias"]
    assert tuple(p2.fc1.weight.shape) == (512, 348) and tuple(p2.log_std.weight.shape) == (17, 512)
    assert abs(p2.action_scale - 0.4) < 1e-12 and p2.action_bias == 0.0


def test_install_registers_reference_module_names(hw):
    import sys
    saved = {k: sys.modules.get(k) for k in ("sac_imp", "replay_buffer", "networks_model1", "networks_model2")}
    try:
        hw.install()
        from sac_imp import SAC
        from replay_buffer import PrioritizedReplayBuffer, ReplayBuffer
        assert SAC is hw.SAC and ReplayBuffer is hw.ReplayBuffer and PrioritizedReplayBuffer is hw.PrioritizedReplayBuffer
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_no_cpu_fallback(hw):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        hw.SAC(8, 2, device="cpu")
    with pytest.raises(RuntimeError):
        hw.SAC(8, 2, device="cuda")
    buf = hw.ReplayBuffer()
    with pytest.raises(RuntimeError):
        buf.push([0.0] * 3, [0.0], 0.0, [0.0] * 3, False)
    assert hw._native.lib().sacb_device_count() == 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "humanoid-walking-with-sac_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the oracle", ""), f


def test_range_sample_is_random_sample(hw):
    """The uniform buffer's index draw: same picks and same consumption of the global `random` stream as
    `random.sample(range(n), k)` (== `random.sample(deque, k)`, replay_buffer.py:15), on the pool path, the set path, with
    rejections (n just above a power of two) and with repeated picks (k close to n)."""
    import random
    from humanoid_walking_with_sac_b200.replay_buffer import _range_sample
    for n, k in [(1_000_000, 256), (5000, 256), (1100, 256), (2 ** 20, 256), (2 ** 20 + 1, 64), (300000, 1024), (1046, 256), (100, 7), (123457, 1), (2000, 1500), (7, 0)]:
        for seed in range(4):
            random.seed(seed)
            ref = random.sample(range(n), k)
            after_ref = random.random()
            random.seed(seed)
            got = _range_sample(n, k)
            assert list(got) == ref and random.random() == after_ref, (n, k, seed)
    with pytest.raises(ValueError):
        _range_sample(10, 11)


def _layout(x):
    """Structure of a checkpoint value as the reference's load code meets it: container types, keys, tensor shapes and dtypes."""
    import collections
    import numpy as np
    import torch
    if torch.is_tensor(x):
        return ("tensor", tuple(x.shape), x.dtype)
    if isinstance(x, np.ndarray):
        return ("ndarray", x.shape)
    if isinstance(x, dict):
        return (type(x).__name__, {k: _layout(v) for k, v in x.items()})
    if isinstance(x, (list, tuple, collections.deque)):
        return (type(x).__name__, [_layout(v) for v in x])
    return type(x).__name__


def test_reference_loads_product_checkpoints():
    """Interop in the other direction: files written by the PRODUCT on a B200 (tests/test_gpu_networks_ckpt.py::
    test_write_product_checkpoints_for_the_reference, committed under tests/golden/) can be resumed by the reference's
    SAC.load / SAC.load_checkpoint (sac_imp.py:164-173, :203-233) and lead to the same next step the product took.
    (1) Every key, container, tensor shape and dtype equals those of the save() / save_checkpoint() pair the reference itself
    wrote after the same two updates (tests/golden/ckpt_ref_*.pt).  (2) The reference's resume and update, as restated by the
    oracle (pinned to the reference resuming its own file: test_oracle_nets_ckpt_golden.py), take the product's third step.
    The losses are the interop evidence; the oracle then steps the temperature like the product, whereas the reference's own
    load_checkpoint (sac_imp.py:222-226) rebinds `log_alpha` away from its optimizer and keeps alpha = exp(loaded log_alpha)."""
    import numpy as np
    import torch
    from oracle import sac_oracle_np as O
    from tests.golden import cases
    from tests.util import state_from_checkpoint
    gold = os.path.join(ROOT, "tests", "golden")
    load = lambda f: torch.load(os.path.join(gold, f), map_location="cpu", weights_only=False)
    for product, reference in (("product_save.pt", "ckpt_ref_save.pt"), ("product_checkpoint.pt", "ckpt_ref_checkpoint.pt")):
        assert _layout(load(product)) == _layout(load(reference)), product
    ck = load("product_checkpoint.pt")
    for key, ref_value in load("ckpt_ref_checkpoint.pt")["q1_optimizer_state_dict"]["param_groups"][0].items():
        assert ck["q1_optimizer_state_dict"]["param_groups"][0][key] == ref_value, key
    assert (ck["episode"], ck["total_steps"]) == (3, 45) and len(ck["replay_buffer"]) == 20
    assert float(ck["q1_optimizer_state_dict"]["state"][0]["step"]) == 2
    case = cases.UPDATE_CASES["tiny_m1"]
    st, _ = state_from_checkpoint(os.path.join(gold, "product_checkpoint.pt"), case)
    np.testing.assert_allclose(st.alpha, float(np.exp(ck["log_alpha"].detach().numpy()[0])), rtol=1e-6)
    b = O.make_batch(case["obs"], case["act"], case["batch"], seed=case["seed"] * 100 + 2)
    info = O.update_parameters(st, b)
    exp = np.load(os.path.join(gold, "product_expected.npz"))
    np.testing.assert_allclose([info["q1_loss"], info["q2_loss"], info["policy_loss"]], exp["next_losses"], rtol=3e-4)
    np.testing.assert_allclose(st.alpha, exp["next_alpha"], rtol=1e-5)
