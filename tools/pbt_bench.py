"""Population-based training costs on one GPU: the C2 x 128 population step (obs 348, act 17, 3 x 512, B = 256, positions and noise
drawn on the device) with one set of hyperparameters for all agents against one set per agent, and the exploit copy of 32 pairs.
The two hyperparameter settings are timed alternately on the same population (switching them rebuilds nothing).  Prints one JSON line.
usage: pbt_bench.py [n_agents] [steps] [rounds]"""
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
OBS, ACT, HID, B, CAP, PAIRS, COPIES = 348, 17, 512, 256, 2048, 32, 20


def timed(fn, n):
    ms = ctypes.c_float()
    N.check(lib.sacb_timer_start(pop._h))
    for _ in range(n):
        fn()
    N.check(lib.sacb_timer_stop(pop._h, ctypes.byref(ms)))
    return ms.value / n


hw.use_networks("model2")
pop = hw.PopulationSAC(A, OBS, ACT, hidden_dim=HID, device="cuda", capacity=CAP, max_batch=B, seed=1)
rng = np.random.RandomState(0)
for a in range(A):
    pop.push_many(a, rng.standard_normal((CAP, OBS)), rng.uniform(-0.4, 0.4, (CAP, ACT)), rng.standard_normal(CAP),
                  rng.standard_normal((CAP, OBS)), (rng.uniform(size=CAP) < 0.01))
i = np.arange(A)
settings = {
    "homogeneous": [dict(lr=3e-4, gamma=0.99, tau=0.005, target_entropy=-float(ACT)) for _ in i],
    "heterogeneous": [dict(lr=float(3e-4 * 10 ** (k / A - 0.5)), gamma=float(0.95 + 0.049 * k / A), tau=float(0.002 + 0.008 * k / A),
                           target_entropy=float(-ACT * (0.5 + k / A))) for k in i],
}
step = lambda: pop.update_parameters(B, sync=False)
for _ in range(3):
    step()
pop.synchronize()
ms = {k: [] for k in settings}
for _ in range(rounds):
    for name, hps in settings.items():
        for a, h in enumerate(hps):
            pop.set_hyperparameters(a, **h)
        step()
        ms[name].append(timed(step, steps))

dst = list(range(A - PAIRS, A))
src = list(range(PAIRS))
p0, p1 = ctypes.c_void_p(), ctypes.c_void_p()
N.check(lib.sacb_tensor_dev(pop._h, 0, N.NET_POLICY, N.SLOT_PARAM, 0, ctypes.byref(p0)))
N.check(lib.sacb_tensor_dev(pop._h, 1, N.NET_POLICY, N.SLOT_PARAM, 0, ctypes.byref(p1)))
span = p1.value - p0.value                      # bytes of one agent's arena span
pop.exploit(dst, src)
pop.synchronize()
copy_ms = timed(lambda: pop.exploit(dst, src), COPIES)
moved = 2 * PAIRS * span                        # read + write

try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    q = "unknown"
print(json.dumps({
    "gpu": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit": q, "n_agents": A, "steps_per_window": steps,
    "ms_per_population_step": {k: [round(x, 4) for x in v] for k, v in ms.items()},
    "ms_per_population_step_median": {k: round(float(np.median(v)), 4) for k, v in ms.items()},
    "exploit": {"pairs": PAIRS, "agent_span_MB": round(span / 1e6, 3), "ms": round(copy_ms, 4), "GB_per_s": round(moved / (copy_ms * 1e-3) / 1e9, 1)},
}))
