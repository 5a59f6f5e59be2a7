"""Prioritized replay in a population: the C2 x 128 population (obs 348, act 17, 3 x 512, B = 256) with 100 000 transitions per agent and
synthetic priorities per agent (as bench.py sets them), timed with CUDA events on the handle's stream:
  (a) sacb_per_sample_all with device-drawn uniforms: one sampler chain of three launches for all agents
  (b) the same work as one sacb_per_sample call per agent (three launches each)
  (c) the population step with prioritized replay: sample -> IS-weighted update -> |TD| write-back (PopulationSAC(replay="per"))
  (d) the uniform population step (positions drawn on the device, SACB_DEVICE_INDICES) on a handle of the same shapes
(c) and (d) are timed alternately.  Prints one JSON line with the GPU name and power limit read in the same run.
usage: population_per_bench.py [n_agents] [steps] [rounds]"""
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import humanoid_walking_with_sac_b200 as hw

N = hw._native
lib = N.lib()
A = int(sys.argv[1]) if len(sys.argv) > 1 else 128
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 3
OBS, ACT, HID, B, CAP = 348, 17, 512, 256, 100000


def timed(h, fn, n):
    ms = ctypes.c_float()
    N.check(lib.sacb_timer_start(h))
    for _ in range(n):
        fn()
    N.check(lib.sacb_timer_stop(h, ctypes.byref(ms)))
    return ms.value / n


def filled(replay):
    pop = hw.PopulationSAC(A, OBS, ACT, hidden_dim=HID, device="cuda", capacity=CAP, max_batch=B, seed=1, replay=replay,
                           **({"per_weighted_loss": True} if replay == "per" else {}))
    rng = np.random.RandomState(0)
    rows = np.zeros((CAP, int(lib.sacb_row_floats(pop._h))), np.float32)      # [s | s2 | a | r | d], padded
    rows[:, :OBS] = rng.standard_normal((CAP, OBS))
    rows[:, OBS:2 * OBS] = rng.standard_normal((CAP, OBS))
    rows[:, 2 * OBS:2 * OBS + ACT] = rng.uniform(-0.4, 0.4, (CAP, ACT))
    rows[:, 2 * OBS + ACT] = rng.standard_normal(CAP)
    rows[:, 2 * OBS + ACT + 1] = rng.uniform(size=CAP) < 0.01
    for a in range(A):
        N.check(lib.sacb_push_rows(pop._h, a, N.ptr(rows), CAP))
        if replay == "per":
            pop.set_priorities(a, (np.abs(np.random.RandomState(1000 + a).standard_normal(CAP)) + 1e-6).astype(np.float32))
    return pop


hw.use_networks("model2")
per = filled("per")
uni = filled("uniform")

sample_all = lambda: N.check(lib.sacb_per_sample_all(per._h, None, B, None, None))


def sample_each():
    for a in range(A):
        N.check(lib.sacb_per_sample(per._h, a, None, B, None, None, None, None, None, None, None))


per_step = lambda: per.update_parameters(B, sync=False)
uni_step = lambda: uni.update_parameters(B, sync=False)
for fn in (sample_all, sample_each, per_step, uni_step):      # programs built, modules loaded
    for _ in range(3):
        fn()
per.synchronize(); uni.synchronize()
ms = {"a_sample_all": [], "b_sample_each": [], "c_per_step": [], "d_uniform_step": []}
for _ in range(rounds):
    ms["a_sample_all"].append(timed(per._h, sample_all, steps))
    ms["b_sample_each"].append(timed(per._h, sample_each, steps))
    ms["c_per_step"].append(timed(per._h, per_step, steps))
    ms["d_uniform_step"].append(timed(uni._h, uni_step, steps))
per.synchronize(); uni.synchronize()
med = {k: float(np.median(v)) for k, v in ms.items()}

try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    q = "unknown"
print(json.dumps({
    "gpu": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit": q, "n_agents": A, "batch": B, "transitions_per_agent": CAP,
    "p_alpha_MB_all_agents": round(A * CAP * 4 / 1e6, 1), "steps_per_window": steps,
    "ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}, "ms_median": {k: round(v, 4) for k, v in med.items()},
    "per_step_over_uniform_step": round(med["c_per_step"] / med["d_uniform_step"], 4),
    "sample_each_over_sample_all": round(med["b_sample_each"] / med["a_sample_all"], 2),
}))
