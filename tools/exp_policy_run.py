"""Agent evaluation three ways, alternated in one process: 16384 episodes of 3-20-10-weighted at k = 2 under a
PairsPolicy with hidden = 128, sampled and greedy.
  policy_run  run_episodes(net) -- bb_run_policy, whole episodes in one launch
  step_api    policy(net, counter=t) + step() until every environment is done -- two launches and a status read per step
  degree      run_episodes('degree') -- the same episodes' count under a built-in rule: what the head costs
Times are CUDA events around the whole call (the step API's host round trips included), L2 flushed (160 MiB write) in
front of every pass.  Also checks that the policy runner and the step API give the same records.  Prints one JSON line.
  python tools/exp_policy_run.py [rounds]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs  # noqa: E402
from deepgroebner_b200.rollout import PairsPolicy  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
E, dist, k, H = 16384, "3-20-10-weighted", 2, 128
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
runner = BuchbergerEngine(dist, k=k, num_envs=resident_envs(0, 3))
stepper = BuchbergerEngine(dist, k=k, num_envs=E)
net = PairsPolicy(runner.cols, hidden=H, torch_seed=1, seed=3)
flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")
fields = ("steps", "additions", "zero_reductions", "nonzero_reductions", "status", "trace_hash")


def policy_run(greedy):
    return runner.run_episodes(net, episodes=E, greedy=greedy, to_host=False)[0]


def step_api(greedy):
    stepper.seed(0)
    stepper.reset()
    t = 0
    while bool((stepper.status() == 1).any()):
        actions, _ = stepper.policy(net, counter=t, greedy=greedy)
        stepper.step(actions)
        t += 1
    return t


def degree(_):
    return runner.run_episodes("degree", episodes=E, to_host=False)[0]


def timed(fn, greedy):
    flush.fill_(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn(greedy)
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


cases = [(n, f, g) for g in (False, True) for n, f in (("policy_run", policy_run), ("step_api", step_api))] + \
        [("degree", degree, False)]
same, steps = {}, {}
for g in (False, True):   # warm-up, and the records of both paths
    rec = runner.run_episodes(net, episodes=E, greedy=g)[0]
    step_api(g)
    st = stepper.stats()
    same[g] = all(np.array_equal(rec[f], st[f]) for f in fields)
    steps[g] = int(rec["steps"].sum())
steps["degree"] = int(runner.run_episodes("degree", episodes=E)[0]["steps"].sum())
ms = {(n, g): [] for n, _, g in cases}
for r in range(rounds):
    for n, f, g in (cases if r % 2 == 0 else cases[::-1]):
        ms[(n, g)].append(timed(f, g))
out = {"gpu": smi, "workload": "%s k=%d H=%d, %d episodes, %d runner slots" % (dist, k, H, E, runner.num_envs),
       "rounds": rounds, "step_api_records_equal": {"sampled": same[False], "greedy": same[True]}}
for (n, g), x in ms.items():
    x = np.array(x)
    s = steps["degree"] if n == "degree" else steps[g]
    out["%s%s" % (n, "" if n == "degree" else ("_greedy" if g else "_sampled"))] = {
        "ms_median": float(np.median(x)), "min": float(x.min()), "max": float(x.max()), "env_steps": s,
        "Msteps_per_s_median": s / float(np.median(x)) / 1e3}
print(json.dumps(out))
