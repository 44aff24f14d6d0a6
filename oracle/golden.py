"""TEST INFRASTRUCTURE ONLY -- stored digests of whole-run episode records (tests/golden/records.json).

The full-size GPU tests and bench.py's parity gate compare every record of a launch with the unmodified reference's
records (oracle/_ref, ``run_records``).  Where oracle/_ref is not built they compare with digests of those records
stored in the repository instead: one SHA-256 per record field over all episodes of the run, keyed by the run's
parameters.  tests/golden/make_records.py writes the file.
"""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "records.json")
FIELDS = ("steps", "additions", "zero_reductions", "nonzero_reductions", "nbasis", "nterms", "status", "rerolls",
          "trace_hash", "basis_hash", "gb_hash", "gb_polys", "gb_terms", "discounted_return")
_cache = {}


def key(dist, selection, count, seed0=0, sel_seed0=0, max_steps=0, **env_kw):
    """Name of a run of `count` episodes (stream seeds seed0 .. seed0 + count - 1, gamma 0.99, reduced basis computed).
    `env_kw` are BuchbergerEnv options that differ from their defaults (elimination, sort_input, sort_reducers)."""
    parts = [dist, selection, "seed0=%d" % seed0, "n=%d" % count]
    if selection == "random":
        parts.append("sel_seed0=%d" % sel_seed0)
    if max_steps:
        parts.append("max_steps=%d" % max_steps)
    parts += ["%s=%s" % (k, env_kw[k]) for k in sorted(env_kw)]
    return "/".join(parts)


def digests(records, fields=FIELDS):
    return {f: hashlib.sha256(np.ascontiguousarray(records[f]).tobytes()).hexdigest() for f in fields}


def runs():
    if "runs" not in _cache:
        with open(PATH) as f:
            _cache["runs"] = json.load(f)["runs"]
    return _cache["runs"]


def have(k):
    return k in runs()


def mismatches(records, k, fields=FIELDS):
    """The fields of `records` (the first len(records) episodes of run `k`) whose digest differs from the stored one."""
    want = runs()[k]
    if len(records) != want["episodes"]:
        raise ValueError("%d records given for run %s of %d episodes" % (len(records), k, want["episodes"]))
    got = digests(records, fields)
    return [f for f in fields if got[f] != want["sha256"][f]]
