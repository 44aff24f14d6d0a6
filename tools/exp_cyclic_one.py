"""Diagnostic (also the command of the k_run_wide ncu captures): n cyclic-6 episodes (seeded Random, stream
seeds seed .. seed + n - 1) on n environment slots under bb_set_wide(mode).  Defaults: the longest of the 1024 episodes of
the bench (seed 1234 + 241, 696 993 additions) alone = the serial chain that bounds a launch containing it.
  python tools/exp_cyclic_one.py [seed] [mode] [n]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from deepgroebner_b200.buchberger import BuchbergerEngine
seed = int(sys.argv[1]) if len(sys.argv) > 1 else 1234 + 241
mode = int(sys.argv[2]) if len(sys.argv) > 2 else -1
n = int(sys.argv[3]) if len(sys.argv) > 3 else 1
eng = BuchbergerEngine("cyclic-6", num_envs=n)
eng.set_wide(mode)
for rep in range(2):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    stats, _ = eng.run_episodes("random", episodes=n, selection_seed=seed)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    print("%.1f ms, %d additions, %d steps, %.3f us per addition of the longest episode" %
          (ms, stats["additions"].sum(), stats["steps"].sum(), ms * 1e3 / stats["additions"].max()))
