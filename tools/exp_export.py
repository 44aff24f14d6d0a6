"""Cost of the polynomial sinks of bb_run_export, A/B in one process with the variants alternated.

configs[1] (16384 episodes of 3-20-10-weighted under Degree, one resident wave of slots, compute_gb on, L2 flushed by a
160 MiB write before every run): no sink, the reduced-basis sink, both sinks.  cyclic-6 under seeded Random selection,
1024 episodes (k_run_wide): no sink, the reduced-basis sink.  Per variant: the runner's device time (CUDA events inside
bb_run_export, bb_set_timing) and the wall time of the whole run_episodes call (records to the host; with sinks also the
fill check and the canonical episode order), median and spread over the repeats, with the card's name, power limit and
maximum SM clock.  Writes the JSON to the path given as the first argument (default exp_export.json)."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs

REPEATS = 7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def measure(eng, variants, flush, **run_kw):
    """{variant: (runner ms list, call ms list)} over REPEATS rounds, the variants alternated within every round."""
    eng.set_timing(True)
    res = {v: ([], []) for v in variants}
    ref = None
    for r in range(REPEATS + 1):   # round 0 warms every variant up
        for v, kw in variants.items():
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = eng.run_episodes(**run_kw, **kw)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            stats = got[0]
            if ref is None:
                ref = stats.tobytes()
            assert stats.tobytes() == ref, v   # a sink never changes a record
            if r:
                res[v][0].append(eng.last_run_ms()[1])
                res[v][1].append(wall)
    return res


def summary(res, base):
    out = {}
    b = float(np.median(res[base][0]))
    for v, (run, call) in res.items():
        out[v] = {"runner_ms_median": float(np.median(run)), "runner_ms_min": float(np.min(run)),
                  "runner_ms_max": float(np.max(run)), "call_ms_median": float(np.median(call)),
                  "runner_vs_%s" % base: float(np.median(run)) / b - 1.0}
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "exp_export.json"
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    line = {"card": card(), "repeats": REPEATS}
    E = 16384
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=min(resident_envs(0, 3), E))
    res = measure(eng, {"no_sink": {}, "gb_sink": dict(return_gb=True), "both_sinks": dict(return_gb=True, return_basis=True)},
                  flush, strategy="degree", episodes=E, compute_gb=True, gamma=0.99)
    line["configs1_3-20-10-weighted_degree_16384"] = summary(res, "no_sink")
    cyc = BuchbergerEngine("cyclic-6", num_envs=1024)
    res = measure(cyc, {"no_sink": {}, "gb_sink": dict(return_gb=True)}, flush, strategy="random", episodes=1024,
                  selection_seed=1234, compute_gb=True, gamma=0.99)
    line["cyclic6_random_1024"] = summary(res, "no_sink")
    with open(path, "w") as fh:
        json.dump(line, fh, indent=1)
    print(json.dumps(line, indent=1))


if __name__ == "__main__":
    main()
