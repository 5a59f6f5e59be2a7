"""A/B timing of the C2 update program (sacb_time_update, CUDA events over graph replays).  usage: ab_update.py [iters]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import humanoid_walking_with_sac_b200 as hw
from tests.golden import cases
from tests.util import batch_of, make_agent
N = hw._native
iters = int(sys.argv[1]) if len(sys.argv) > 1 else 300
launch = sys.argv[2] if len(sys.argv) > 2 else "staged"
case = cases.UPDATE_CASES["c2_humanoid_m2"]
agent, st = make_agent(hw, case, math="bf16x3", launch=launch)
agent.update_from_batch(batch_of(case, 0))
best = 1e9
for rep in range(5):
    ms = ctypes.c_float()
    N.check(N.lib().sacb_time_update(agent._h, 256, iters, ctypes.byref(ms)))
    best = min(best, ms.value)
print(f"AB_UPDATE launch={launch} env={os.environ.get('SACB_AB_TAG', '')} best_ms={best:.4f} stages={agent.stats()['n_stages']}")
