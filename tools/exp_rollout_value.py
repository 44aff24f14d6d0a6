"""PPO trajectories with a Degree value baseline: the fused rollout with values against the step-API loop it replaces.

Workload: 3-20-10-weighted, LeadMonomialsEnv(k=2), PMLP head H = 128, N = 16384 environments, T = 64 steps, auto-reset on,
value('degree', 0.99) of every state.  Three arms, each timed with CUDA events around the whole T-step window:
  fused  -- one bb_rollout_value launch;
  loop   -- per step bb_value, bb_policy_pmlp(counter0 + t), bb_step (what a caller writes without bb_rollout_value);
  floor  -- bb_rollout without values.
Every arm starts from the same reseeded, reset environments.  The arms alternate within each repetition, after a warm-up
repetition; the fused and loop arms must agree bit for bit (values, NaN included; actions, log-probabilities, rewards and
done flags of the running steps; lengths).  Prints the card name and power limit, one JSON line per repetition and one
with the medians.

    python tools/exp_rollout_value.py [--reps 5] [--warmup 1] [--envs 16384] [--steps 64]
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
from deepgroebner_b200.rollout import PairsPolicy  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def restart(env, N):
    env.seed(np.arange(1000, 1000 + N))
    env.engine.reset()
    torch.cuda.synchronize()


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=64)
    args = ap.parse_args()
    N, T, C0 = args.envs, args.steps, 1000
    print("card:", card(), flush=True)
    envs = {arm: LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=128) for arm in ("fused", "loop", "floor")}
    for env in envs.values():
        env.engine.set_auto_reset(True)
    net = PairsPolicy(envs["fused"].engine.cols, 128, torch_seed=1, seed=7, device="cuda")
    dev = envs["loop"].engine.device
    lv = torch.empty((T, N), dtype=torch.float64, device=dev)
    ll, la = torch.empty((T, N), dtype=torch.int32, device=dev), torch.empty((T, N), dtype=torch.int32, device=dev)
    lp, lr = torch.empty((T, N), dtype=torch.float32, device=dev), torch.empty((T, N), dtype=torch.float64, device=dev)
    ld = torch.empty((T, N), dtype=torch.uint8, device=dev)

    def fused():
        return envs["fused"].engine.rollout(net, T, counter0=C0, value="degree", value_gamma=0.99)

    def loop():
        eng = envs["loop"].engine
        for t in range(T):
            eng.value("degree", 0.99, out=lv[t])
            ll[t].copy_(eng.lengths())
            a, p = eng.policy(net, counter=C0 + t)
            la[t].copy_(a)
            lp[t].copy_(p)
            eng.step(a, reward=lr[t], done=ld[t])

    def floor():
        return envs["floor"].engine.rollout(net, T, counter0=C0)

    arms = [("fused", fused), ("loop", loop), ("floor", floor)]
    ms = {a: [] for a, _ in arms}
    for rep in range(args.warmup + args.reps):
        order = arms if rep % 2 == 0 else arms[::-1]
        got = {}
        for name, fn in order:
            restart(envs[name], N)
            t, got[name] = timed(fn)
            if rep >= args.warmup:
                ms[name].append(t)
        f = got["fused"]
        run = f["actions"] >= 0
        same = (np.array_equal(f["value"].view(torch.int64).cpu().numpy(), lv.t().contiguous().view(torch.int64).cpu().numpy())
                and torch.equal(f["lengths"], ll.t()) and torch.equal(run, ll.t() > 0)
                and torch.equal(f["actions"][run], la.t()[run]) and torch.equal(f["logp"][run], lp.t()[run])
                and torch.equal(f["reward"][run], lr.t()[run].to(torch.float32)) and torch.equal(f["done"][run], ld.t()[run]))
        assert same, "fused and step-API loop differ in repetition %d" % rep
        assert torch.equal(f["actions"], got["floor"]["actions"]) and torch.equal(f["reward"], got["floor"]["reward"])
        if rep >= args.warmup:
            print(json.dumps(dict(rep=rep - args.warmup, **{n + "_ms": round(ms[n][-1], 3) for n, _ in arms},
                                  fused_equals_loop=True)), flush=True)
    med = {a: float(np.median(v)) for a, v in ms.items()}
    v = f["value"]
    print(json.dumps(dict(workload="3-20-10-weighted k=2 H=128 value=degree gamma=0.99", envs=N, steps=T, reps=args.reps,
                          fused_ms=round(med["fused"], 3), loop_ms=round(med["loop"], 3), floor_ms=round(med["floor"], 3),
                          loop_over_fused=round(med["loop"] / med["fused"], 3),
                          fused_over_floor=round(med["fused"] / med["floor"], 3),
                          env_steps_per_s_fused=round(N * T / med["fused"] * 1e3),
                          value_nan=int(torch.isnan(v).sum()), fused_equals_loop=True)), flush=True)


if __name__ == "__main__":
    main()
