"""Throughput of bb_reduce (reduce(g, F) on the device) on the reduced bases of a whole run.

Workload: the 16384 reduced Groebner bases of 3-20-10-weighted under Degree selection, computed on the device by
run_episodes(return_gb=True), each the divisor list of 1 or 16 random dividends (8 random terms before duplicates are
dropped, exponents 0..12, queries of one basis adjacent).  Each configuration is timed with CUDA events around every
bb_reduce launch, once with a remainder sink and once without; the L2 cache is overwritten before every timed launch.
Prints the card name and power limit, then one JSON line per configuration.

    python tools/exp_reduce.py [--launches 20] [--warmup 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepgroebner_b200.buchberger import BuchbergerEngine, _ptr, _stream  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def random_queries(rng, nlists, per, terms=8, emax=12):
    """per dividends per list, list-major; terms strictly descending in grevlex (ascending packed key, 3 variables)."""
    Q = nlists * per
    e = rng.integers(0, emax + 1, size=(Q, terms, 3)).astype(np.int64)
    key = e[..., 0] | (e[..., 1] << 16) | (e[..., 2] << 32) | ((32767 - e.sum(-1)) << 48)
    key = np.sort(key, axis=1)
    keep = np.ones_like(key, bool)
    keep[:, 1:] = key[:, 1:] != key[:, :-1]
    k = key[keep]
    exps = np.stack([k & 0xffff, (k >> 16) & 0xffff, (k >> 32) & 0xffff], 1).astype(np.int32)
    offsets = np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64)
    coefs = rng.integers(1, 32003, size=len(k)).astype(np.int32)
    which = np.repeat(np.arange(nlists, dtype=np.int32), per)
    return offsets, exps, coefs, which


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=3552)
    stats, _, out = eng.run_episodes("degree", episodes=16384, return_gb=True)
    gb = out["gb"]
    assert bool(gb.stored.all()), "every basis of the workload is stored"
    dev = eng.device
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # twice the L2
    rng = np.random.default_rng(0)
    for per in (1, 16):
        q_off, q_ex, q_cf, which = (torch.as_tensor(a, device=dev) for a in random_queries(rng, len(gb), per))
        Q = which.numel()
        steps, rlen, status = (torch.empty(Q, dtype=torch.int32, device=dev) for _ in range(3))
        for with_sink in (True, False):
            sink = eng._sink(Q, Q, 4 * q_cf.numel()) if with_sink else None
            times = []
            for it in range(args.warmup + args.launches):
                if sink:
                    sink[0]["used"].zero_()
                flush.fill_(it & 0xff)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                rc = eng.lib.bb_reduce(eng.h, len(gb), _ptr(gb.ep_offsets), _ptr(gb.poly_offsets), _ptr(gb.exps), _ptr(gb.coefs),
                                       Q, _ptr(q_off), _ptr(q_ex), _ptr(q_cf), _ptr(which), 1, _ptr(steps), _ptr(rlen),
                                       _ptr(status), sink[1] if sink else None, _stream())
                b.record()
                assert rc == 0, eng.lib.bb_last_error(eng.h)
                torch.cuda.synchronize()
                if it >= args.warmup:
                    times.append(a.elapsed_time(b))
            assert bool((status == 2).all())
            if sink:
                assert sink[0]["used"].tolist()[2] == 0
            ms = float(np.median(times))
            adds = int(steps.sum())
            print(json.dumps(dict(queries_per_basis=per, queries=Q, sink=with_sink, launches=len(times), l2_flushed=True,
                                  ms_median=round(ms, 4), ms_min=round(min(times), 4), ms_max=round(max(times), 4),
                                  queries_per_s=round(Q / ms * 1e3), additions=adds,
                                  additions_per_s=round(adds / ms * 1e3), remainder_terms=int(rlen.sum()))), flush=True)


if __name__ == "__main__":
    main()
