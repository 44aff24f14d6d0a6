"""ctypes binding of libbbenv.so (C-ABI declared in include/bbenv.h).

There is NO CPU fallback: if the CUDA library is missing, cannot be loaded, or no CUDA device is present, the
import of the product path fails loudly.  Nothing here (or anywhere under deepgroebner_b200/) touches oracle/.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# BBENV_LIB selects another build of the SAME library (A/B runs of kernel variants); it is never a fallback.
LIB_PATH = os.environ.get("BBENV_LIB") or os.path.join(HERE, "libbbenv.so")

BB_ABI_VERSION = 3

ELIMINATION = {"gebauermoeller": 0, "lcm": 1, "none": 2}
REWARDS = {"additions": 0, "reductions": 1}
SELECTION = {"first": 0, "degree": 1, "normal": 2, "sugar": 3, "random": 4, "last": 5, "codegree": 6, "strange": 7,
             "spice": 8}
VALUE_SAMPLE = 100  # bb_value only: value("sample")
DISTRIBUTION = {"uniform": 0, "weighted": 1, "maximum": 2}

STATUS_NAMES = {0: "empty", 1: "running", 2: "done", 3: "bad_action", 4: "overflow_basis", 5: "overflow_pairs",
                6: "overflow_terms", 7: "overflow_exponent", 8: "overflow_scratch", 9: "truncated"}
STATUS_COUNT = 10


class BBConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "abi_version", "device", "nvars", "k", "prime", "elimination", "rewards", "sort_input", "sort_reducers",
        "num_envs", "max_basis", "max_pairs", "max_terms", "max_poly_terms", "max_gens", "max_gen_terms")]


class BBCounters(C.Structure):
    _fields_ = [(n, C.c_ulonglong) for n in (
        "env_steps", "additions", "terms_read", "terms_written", "lms_scanned", "term_moves", "update_basis",
        "update_pairs", "obs_rows", "nonzero_reductions", "zero_reductions", "episodes")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class BBEpisodeStats(C.Structure):
    _fields_ = [("steps", C.c_int32), ("additions", C.c_int32), ("zero_reductions", C.c_int32),
                ("nonzero_reductions", C.c_int32), ("nbasis", C.c_int32), ("nterms", C.c_int32),
                ("status", C.c_int32), ("rerolls", C.c_int32), ("trace_hash", C.c_uint64),
                ("basis_hash", C.c_uint64), ("gb_hash", C.c_uint64), ("gb_polys", C.c_int32),
                ("gb_terms", C.c_int32), ("discounted_return", C.c_double)]


class BBPolySink(C.Structure):
    """bb_poly_sink: a packed, caller-owned device buffer of polynomials (bb_run_export)."""
    _fields_ = [("lens_dev", C.c_void_p), ("exps_dev", C.c_void_p), ("coefs_dev", C.c_void_p), ("where_dev", C.c_void_p),
                ("used_dev", C.c_void_p), ("cap_polys", C.c_int64), ("cap_terms", C.c_int64)]


# numpy view of bb_episode_stats (same layout; checked against sizeof in load())
STATS_DTYPE = [("steps", "<i4"), ("additions", "<i4"), ("zero_reductions", "<i4"), ("nonzero_reductions", "<i4"),
               ("nbasis", "<i4"), ("nterms", "<i4"), ("status", "<i4"), ("rerolls", "<i4"), ("trace_hash", "<u8"),
               ("basis_hash", "<u8"), ("gb_hash", "<u8"), ("gb_polys", "<i4"), ("gb_terms", "<i4"),
               ("discounted_return", "<f8")]

EXPORTS = [
    "bb_abi_version", "bb_resident_envs", "bb_create", "bb_destroy", "bb_last_error", "bb_cols", "bb_num_envs", "bb_sm_count",
    "bb_set_distribution", "bb_set_distribution_poly", "bb_seed", "bb_set_ideals", "bb_reset", "bb_step", "bb_select", "bb_observe", "bb_pairs",
    "bb_status", "bb_stats", "bb_run", "bb_download_basis", "bb_final_gb", "bb_counters_read", "bb_hash_item",
    "bb_seed_selection", "bb_value", "bb_copy_env", "bb_set_auto_reset", "bb_step_observe", "bb_step_host", "bb_reset_host", "bb_observe_host", "bb_set_wide", "bb_set_prepare_mode", "bb_set_two_term", "bb_set_selection_seed_stride", "bb_policy_pmlp", "bb_rollout",
    "bb_seed_on", "bb_prepare", "bb_set_episode_offset", "bb_set_timing", "bb_last_run_ms", "bb_set_max_episode_length",
    "bb_set_compaction", "bb_compact", "bb_status_summary", "bb_set_obs_nvars", "bb_discount", "bb_set_serve", "bb_set_prefetch",
    "bb_run_export", "bb_reduce", "bb_run_policy", "bb_rollout_value", "bb_rollout_rows",
]

_lib = None


class BBError(RuntimeError):
    pass


def load():
    """Loads libbbenv.so and declares every prototype.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BBError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(nvcc, sm_100a).  deepgroebner_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, ip, i = C.c_void_p, C.POINTER(C.c_int32), C.c_int
    lib.bb_abi_version.restype = i
    lib.bb_create.restype = i
    lib.bb_create.argtypes = [C.POINTER(BBConfig), C.POINTER(vp)]
    lib.bb_destroy.restype = None
    lib.bb_destroy.argtypes = [vp]
    lib.bb_last_error.restype = C.c_char_p
    lib.bb_last_error.argtypes = [vp]
    for n in ("bb_cols", "bb_num_envs", "bb_sm_count"):
        getattr(lib, n).restype = i
        getattr(lib, n).argtypes = [vp]
    lib.bb_resident_envs.restype = i
    lib.bb_resident_envs.argtypes = [i, i]
    lib.bb_set_distribution.restype = i
    lib.bb_set_distribution.argtypes = [vp, i, i, i, i, i, i]
    lib.bb_set_distribution_poly.restype = i
    lib.bb_set_distribution_poly.argtypes = [vp, i, i, C.c_double, i, i, i]
    lib.bb_seed.restype = i
    lib.bb_seed.argtypes = [vp, ip, i]
    lib.bb_seed_selection.restype = i
    lib.bb_seed_selection.argtypes = [vp, ip, i]
    lib.bb_set_ideals.restype = i
    lib.bb_set_ideals.argtypes = [vp, ip, i, ip, ip, ip, ip]
    lib.bb_reset.restype = i
    lib.bb_reset.argtypes = [vp, vp, vp]
    lib.bb_step.restype = i
    lib.bb_step.argtypes = [vp, vp, vp, vp, vp]
    lib.bb_step_observe.restype = i
    lib.bb_step_observe.argtypes = [vp, vp, vp, vp, vp, vp, i, vp]
    lib.bb_step_host.restype = i
    lib.bb_step_host.argtypes = [vp, vp, vp, vp, vp, vp, i, i, vp]
    lib.bb_reset_host.restype = i
    lib.bb_reset_host.argtypes = [vp, vp, vp, i, i, vp]
    lib.bb_observe_host.restype = i
    lib.bb_observe_host.argtypes = [vp, vp, vp, i, i, vp]
    lib.bb_select.restype = i
    lib.bb_select.argtypes = [vp, i, vp, vp]
    lib.bb_observe.restype = i
    lib.bb_observe.argtypes = [vp, vp, vp, i, vp]
    lib.bb_pairs.restype = i
    lib.bb_pairs.argtypes = [vp, vp, vp, i, vp]
    lib.bb_status.restype = i
    lib.bb_status.argtypes = [vp, vp, vp]
    lib.bb_stats.restype = i
    lib.bb_stats.argtypes = [vp, vp, vp]
    lib.bb_run.restype = i
    lib.bb_run.argtypes = [vp, i, i, i, vp, i, i, C.c_double, i, vp, vp, i, i, vp]
    lib.bb_run_export.restype = i
    lib.bb_run_export.argtypes = lib.bb_run.argtypes + [C.POINTER(BBPolySink), C.POINTER(BBPolySink)]
    lib.bb_reduce.restype = i
    lib.bb_reduce.argtypes = [vp, i, vp, vp, vp, vp, i, vp, vp, vp, vp, i, vp, vp, vp, C.POINTER(BBPolySink), vp]
    lib.bb_value.restype = i
    lib.bb_value.argtypes = [vp, i, C.c_double, i, i, i, vp, vp]
    lib.bb_copy_env.restype = i
    lib.bb_copy_env.argtypes = [vp, i, vp, i, vp]
    lib.bb_set_auto_reset.restype = i
    lib.bb_set_auto_reset.argtypes = [vp, i]
    lib.bb_set_wide.restype = i
    lib.bb_set_wide.argtypes = [vp, i]
    lib.bb_set_prepare_mode.restype = i
    lib.bb_set_prepare_mode.argtypes = [vp, i]
    lib.bb_set_two_term.restype = i
    lib.bb_set_two_term.argtypes = [vp, i]
    lib.bb_set_selection_seed_stride.restype = i
    lib.bb_set_selection_seed_stride.argtypes = [vp, i]
    lib.bb_seed_on.restype = i
    lib.bb_seed_on.argtypes = [vp, ip, i, i, vp]
    lib.bb_prepare.restype = i
    lib.bb_prepare.argtypes = [vp, i, i, vp, vp]
    for n in ("bb_set_episode_offset", "bb_set_timing", "bb_set_max_episode_length", "bb_set_compaction", "bb_set_obs_nvars",
              "bb_set_serve", "bb_set_prefetch"):
        getattr(lib, n).restype = i
        getattr(lib, n).argtypes = [vp, i]
    lib.bb_last_run_ms.restype = i
    lib.bb_last_run_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.bb_compact.restype = i
    lib.bb_compact.argtypes = [vp, vp, vp]
    lib.bb_status_summary.restype = i
    lib.bb_status_summary.argtypes = [vp, ip, vp]
    lib.bb_discount.restype = i
    lib.bb_discount.argtypes = [vp, i, i, vp, vp, C.c_double, vp, vp]
    u64 = C.c_uint64
    lib.bb_policy_pmlp.restype = i
    lib.bb_policy_pmlp.argtypes = [vp, i, vp, vp, vp, vp, u64, u64, i, vp, vp, vp, i, vp]
    lib.bb_rollout.restype = i
    lib.bb_rollout.argtypes = [vp, i, vp, vp, vp, vp, u64, u64, i, i, vp, vp, vp, vp, vp, vp, i, vp]
    lib.bb_rollout_value.restype = i
    lib.bb_rollout_value.argtypes = lib.bb_rollout.argtypes[:-1] + [i, C.c_double, i, i, i, vp, vp]
    lib.bb_rollout_rows.restype = i
    lib.bb_rollout_rows.argtypes = lib.bb_rollout_value.argtypes[:-1] + [vp, C.c_int64, vp]
    lib.bb_run_policy.restype = i
    lib.bb_run_policy.argtypes = [vp, i, vp, vp, vp, vp, u64, u64, i, i, i, vp, i, C.c_double, i, vp, vp, i, i, vp,
                                  C.POINTER(BBPolySink), C.POINTER(BBPolySink)]
    lib.bb_download_basis.restype = i
    lib.bb_download_basis.argtypes = [vp, i, ip, i, ip, ip, i, C.POINTER(C.c_int)]
    lib.bb_final_gb.restype = i
    lib.bb_final_gb.argtypes = [vp, i, ip, i, ip, ip, i, C.POINTER(C.c_int)]
    lib.bb_counters_read.restype = i
    lib.bb_counters_read.argtypes = [vp, C.POINTER(BBCounters), i]
    lib.bb_hash_item.restype = C.c_uint64
    lib.bb_hash_item.argtypes = [C.c_uint64, C.c_uint64]
    if lib.bb_abi_version() != BB_ABI_VERSION:
        raise BBError("libbbenv.so ABI version mismatch")
    import numpy as np
    assert np.dtype(STATS_DTYPE).itemsize == C.sizeof(BBEpisodeStats)
    _lib = lib
    return lib


def check(lib, handle, rc, what):
    if rc < 0:
        msg = lib.bb_last_error(handle)
        raise BBError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
    return rc
