"""Writes tests/golden/records.json: per-field SHA-256 digests of the whole-run episode records (bb_episode_stats
layout) that the full-size GPU tests and bench.py's parity gate compare with when oracle/_ref is not built.

    python tests/golden/make_records.py

Every run is computed by the unmodified reference (oracle/_ref, ref_run_records) when it is built, otherwise by the C
restatement (oracle/bb_oracle.c) on all host cores, episode by episode through its BuchbergerEnv.
"""
import json
import os
import sys
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import golden  # noqa: E402
from oracle import oracle as O  # noqa: E402

# (dist, selection, count, run options): the runs of tests/test_gpu_parity.py, tests/test_gpu_round2.py,
# tests/test_gpu_nccl.py and bench.py
RUNS = [("3-20-10-weighted", s, 16384, {}) for s in ("degree", "first", "normal")]
RUNS += [(d, "degree", 65536, {}) for d in ("3-20-10-uniform", "5-5-10-uniform")]
RUNS += [("cyclic-6", "random", n, dict(sel_seed0=1234)) for n in (256, 1024)]
RUNS += [(d, "normal", 600, dict(seed0=11, max_steps=400, **kw)) for d, kw in (
    ("3-20-10-weighted", {}), ("5-5-10-uniform", {}), ("3-12-6-weighted-pure", dict(sort_reducers=False)),
    ("3-4-16-uniform", {}), ("2-3-3-weighted", {}))]
RUNS += [(d, s, 2048, dict(seed0=3)) for d in ("7-2-5-uniform", "8-2-5-uniform", "8-3-4-uniform") for s in ("normal", "degree")]
RUNS += [("3-20-10-weighted", "degree", n, dict(seed0=b)) for n, bases in ((3000, (0, 5000, 9000)), (6000, (0, 7000, 14000)))
         for b in bases]
RUNS += [("3-20-10-uniform", "random", 157, dict(seed0=10, sel_seed0=77))]
RUNS += [("3-20-10-weighted", s, 1001, dict(seed0=20, sel_seed0=5)) for s in ("degree", "random")]
CHUNK = 64


class Minstd:
    """std::default_random_engine (minstd_rand0) and choice()'s uniform_int_distribution, as oracle/bb_oracle.c."""

    def __init__(self, seed):
        self.x = (seed % 2147483647) or 1

    def index(self, size):
        scaling = 2147483645 // size
        while True:
            self.x = self.x * 16807 % 2147483647
            if self.x - 1 < size * scaling:
                return (self.x - 1) // scaling


def port_records(dist, selection, seed0, count, sel_seed0=0, max_steps=0, gamma=0.99, **env_kw):
    """Records of episodes seed0 .. seed0 + count - 1 from the C restatement, as ref_run_records computes them
    (Random: choice() on minstd_rand0 seeded sel_seed0 + e)."""
    from hashing import polys_hash, trace_hash
    if env_kw.get("sort_input"):
        raise NotImplementedError("re-rolls are counted on the unsorted generator output")
    port = O.load_port()
    env = port.env(dist, **env_kw)
    gen = port.generator(dist)
    out = np.zeros(count, dtype=np.dtype(O.Oracle.RECORD_DTYPE))
    for e in range(count):
        env.seed(seed0 + e)
        G0, _ = env.reset()
        gen.seed(seed0 + e)
        rolls = 0
        while gen.next() != G0 and rolls <= 1000:   # reset() draws again while the pair set is empty
            rolls += 1
        if max_steps or selection == "random":
            rows = []
            rng = Minstd(sel_seed0 + e)
            while env.pairs() and (not max_steps or len(rows) < max_steps):
                P = env.pairs()
                p = P[rng.index(len(P)) if selection == "random" else env.select(selection)]
                reward, _ = env.step(p)
                rows.append([p[0], p[1], int(-reward)])
            t = np.array(rows, np.int32).reshape(-1, 3)
        else:
            t = env.run(selection=selection)[:, :3]
        done = not env.pairs()
        B = env.basis()
        r = out[e]
        r["steps"], r["additions"], r["nbasis"] = len(t), int(t[:, 2].sum()), len(B)
        r["nterms"] = sum(len(g) for g in B)
        r["nonzero_reductions"] = len(B) - len(G0)
        r["zero_reductions"] = len(t) - r["nonzero_reductions"]
        r["status"], r["rerolls"] = (2 if done else 1), rolls
        r["trace_hash"], r["basis_hash"] = trace_hash(t), polys_hash(B)
        if done:
            gb = env.final_gb()
            r["gb_hash"], r["gb_polys"], r["gb_terms"] = polys_hash(gb), len(gb), sum(len(g) for g in gb)
        ret, disc = 0.0, 1.0
        for a in t[:, 2]:
            ret += disc * -float(a)
            disc *= gamma
        r["discounted_return"] = ret
    return out


def _chunk(job):
    dist, selection, kw, lo, hi = job
    kw = dict(kw)
    return port_records(dist, selection, kw.pop("seed0", 0) + lo, hi - lo, sel_seed0=kw.pop("sel_seed0", 0) + lo, **kw)


def main():
    out = {}
    ref = O.load_ref() if O.have_ref() else None
    with Pool() as pool:
        for dist, selection, count, kw in RUNS:
            k = golden.key(dist, selection, count, **kw)
            if ref is not None:
                rec = ref.run_records(dist, selection, count, gamma=0.99, compute_gb=True, **kw)
                source = "unmodified reference (oracle/_ref run_records)"
            else:
                jobs = [(dist, selection, kw, lo, min(count, lo + CHUNK)) for lo in range(0, count, CHUNK)]
                rec = np.concatenate(pool.map(_chunk, jobs, chunksize=1))
                source = "C restatement (oracle/bb_oracle.c), BuchbergerEnv stepped episode by episode"
            out[k] = {"episodes": count, "source": source, "sha256": golden.digests(rec),
                      "totals": {"steps": int(rec["steps"].sum()), "additions": int(rec["additions"].sum())}}
            print(k, out[k]["totals"], flush=True)
    with open(golden.PATH, "w") as f:
        json.dump({"runs": out}, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
