"""A/B of the two-term runner (bb_set_two_term) against the general one on bench.py's flagship workload, in one process:
16384 episodes of 3-20-10-weighted under Degree, alternated launches, k_run time from the CUDA events inside bb_run
(bb_set_timing), L2 flushed (160 MiB write) in front of every launch.  Also checks that both give the same records and
counters.  Prints one JSON line.
  python tools/exp_two_term.py [rounds] [dist] [strategy] [episodes]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 7
dist = sys.argv[2] if len(sys.argv) > 2 else "3-20-10-weighted"
strategy = sys.argv[3] if len(sys.argv) > 3 else "degree"
E = int(sys.argv[4]) if len(sys.argv) > 4 else 16384
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
eng = BuchbergerEngine(dist, num_envs=min(E, resident_envs(0, int(dist.split("-")[0]))))
flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")


def launch(two, timed=True):
    eng.set_two_term(two)
    eng.set_timing(timed)
    flush.fill_(1)
    stats, _ = eng.run_episodes(strategy, episodes=E, selection_seed=0, gamma=0.99)
    return stats, (eng.last_run_ms()[1] if timed else None)


recs, ctrs = {}, {}
for two in (True, False):   # warm-up, and the results of both
    eng.counters(reset=True)
    recs[two], _ = launch(two, timed=False)
    ctrs[two] = eng.counters(reset=True)
ms = {True: [], False: []}
for r in range(rounds):
    for two in ((True, False) if r % 2 == 0 else (False, True)):
        ms[two].append(launch(two)[1])
steps = int(recs[True]["steps"].sum())
out = {"gpu": smi, "workload": "%s %s %d episodes, %d slots" % (dist, strategy, E, eng.num_envs), "rounds": rounds,
       "env_steps_per_launch": steps, "identical_records": recs[True].tobytes() == recs[False].tobytes(),
       "identical_counters": ctrs[True] == ctrs[False]}
for two, name in ((True, "two_term"), (False, "general")):
    x = np.array(ms[two])
    out[name] = {"k_run_ms_median": float(np.median(x)), "min": float(x.min()), "max": float(x.max()),
                 "Msteps_per_s_median": steps / float(np.median(x)) / 1e3, "all_ms": [round(float(v), 4) for v in x]}
out["speedup_median"] = out["general"]["k_run_ms_median"] / out["two_term"]["k_run_ms_median"]
print(json.dumps(out))
