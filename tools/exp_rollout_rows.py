"""PPO training states stored at their own row count (bb_rollout_rows) against the dense [N, T, pmax, cols] block.

Workloads: 3-20-10-weighted and 5-5-10-uniform, LeadMonomialsEnv(k=2), PMLP head H = 128, N = 16384 environments,
T = 64 steps, auto-reset on.  Arms, each one fused rollout launch timed with CUDA events:
  none      -- no states stored (the floor);
  dense64   -- obs at pmax = 64 (rollout()'s default): bytes, and the states wider than 64 rows, which are lost;
  densemax  -- obs at pmax = the largest |P| the none arm saw: bytes;
  rows      -- the row store at the default budget max(max_pairs, 64 T): bytes, halted environments, rows used per
               environment (median, max);
  rowsbig   -- the row store at T x (largest |P|) rows per environment, which cannot halt: the same figures.
Every arm starts from the same reseeded, reset environments, so all play the same trajectories (a halted environment
plays the same prefix); this is checked.  The arms rotate within each repetition, after a warm-up repetition.  Prints
the card name and power limit, one JSON line per repetition and one per workload with the medians.

    python tools/exp_rollout_rows.py [--reps 5] [--warmup 1] [--envs 16384] [--steps 64] [--dists a,b]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepgroebner_b200 import LeadMonomialsEnv  # noqa: E402
from deepgroebner_b200.rollout import PairsPolicy, TrajectoryBatch  # noqa: E402

TRAJ = ("actions", "logp", "reward", "done", "lengths")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def workload(dist, N, T, reps, warmup):
    env = LeadMonomialsEnv(dist, k=2, num_envs=N, pmax=64)
    eng = env.engine
    eng.set_auto_reset(True)
    net = PairsPolicy(eng.cols, 128, torch_seed=1, seed=7, device="cuda")
    C0 = 1000

    def run(**kw):
        env.seed(np.arange(1000, 1000 + N))
        eng.reset()
        torch.cuda.synchronize()
        return timed(lambda: eng.rollout(net, T, counter0=C0, **kw))

    _, ref = run()
    pwide = int(ref["lengths"].max())
    default_rows = max(eng.caps["max_pairs"], eng.ROWS_PER_STEP * T)
    arms = {"none": {}, "dense64": dict(store_obs=True, pmax=64), "densemax": dict(store_obs=True, pmax=pwide),
            "rows": dict(rows_per_env=True), "rowsbig": dict(rows_per_env=T * pwide)}
    ms = {a: [] for a in arms}
    facts = {}
    names = list(arms)
    for rep in range(warmup + reps):
        for name in names[rep % len(names):] + names[:rep % len(names)]:
            t, out = run(**arms[name])
            took = out["actions"] >= 0
            for n in TRAJ:   # the same trajectories in every arm; a halted environment plays the same prefix
                assert torch.equal(out[n][took], ref[n][took]), (name, n)
            if rep >= warmup:
                ms[name].append(t)
            if name in facts:
                del out
                continue
            f = {}
            if "obs" in out:
                f["bytes"] = out["obs"].numel() * 4
                f["wide_states"] = int((took & (out["lengths"] > out["obs"].shape[2])).sum())
                tb = TrajectoryBatch(out)
                tb.get()
                f["dropped_wide"] = tb.dropped_wide
            if "rows" in out:
                tb = TrajectoryBatch(out)
                used = (out["lengths"].to(torch.int64) * took).sum(dim=1).double()
                f.update(bytes=out["rows"].numel() * 4, rows_per_env=out["rows"].shape[1], halted=tb.halted,
                         rows_used_median=float(used.median()), rows_used_max=int(used.max()),
                         training_samples=len(tb.get()[1]))
            facts[name] = f
            del out
        if rep >= warmup:
            print(json.dumps(dict(workload=dist, rep=rep - warmup, **{n + "_ms": round(v[-1], 3) for n, v in ms.items()})),
                  flush=True)
    mean_rows = float(ref["lengths"][ref["actions"] >= 0].double().mean())
    print(json.dumps(dict(workload="%s k=2 H=128" % dist, envs=N, steps=T, reps=reps, largest_P=pwide,
                          mean_rows_per_state=round(mean_rows, 2), default_rows_per_env=default_rows,
                          arms={a: dict(ms=round(float(np.median(ms[a])), 3), **facts.get(a, {})) for a in arms})), flush=True)
    del env, eng
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--dists", default="3-20-10-weighted,5-5-10-uniform")
    args = ap.parse_args()
    print("card:", card(), flush=True)
    for dist in args.dists.split(","):
        workload(dist, args.envs, args.steps, args.reps, args.warmup)


if __name__ == "__main__":
    main()
