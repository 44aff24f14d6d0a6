#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched Buchberger environment on B200 (BASELINE.json metric), beside the
reference's own CPU environment.

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's CUDA path
  python bench.py --impl reference [--steps K] [--warmup W]      the unmodified reference on the host cores
  BB_BENCH_WORKLOAD=u3|u5|cyclic6|rollout python bench.py ...    another BASELINE config (same as --workload)

Workload (BASELINE.json configs[1]): 3-20-10-weighted, 16384 episodes per GPU run to completion under Degree
selection; episode e draws its ideal from the reference generator stream seed(e).  One bench "step" = one pass of
the hot path over that batch: episode preparation (ideal generator + reset, k_prepare_lanes + k_order) and the
persistent episode runner (k_run: select + spoly + reduce + update for every step of every episode).  Steps are
pipelined the way a job of many batches runs: the batch of step i + 1 is prepared on a side stream while the runner
works through batch i (bb_prepare, two staging sets); both lie inside the CUDA-event pair of step i.
`value` = env steps / device time with the inputs (seeds) resident in HBM; `e2e` = the same through
BuchbergerEngine.prepare_episodes / run_episodes with HOST buffers (pinned seeds H2D, episode records D2H and a
stream synchronisation per step, inside the timed region).

Parity gate: EVERY episode record of the timed output (and of one extra launch with the reduced Groebner basis,
outside the timed region) is compared with the unmodified reference (oracle/_ref, ref_run_records) -- pair sequence and
per-step rewards (rolling checksum), length, additions, final basis, reduced basis, discounted return -- or, where
oracle/_ref is not built, with the stored digests of those records (tests/golden/records.json).  A mismatch aborts the
run: no `value` is printed.  The oracle / reference is used as the checker, the cpu_baseline leg and the
`--impl reference` arm only -- never inside a timed GPU region.  --dump-outputs DIR writes what the last timed step
computed (the episode records) as .npy files, so that two builds can be compared output for output.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
# version banner there under torchrun), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a
# private duplicate of the original stdout.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


DIST = "3-20-10-weighted"
STRATEGY = "degree"
EPISODES = 16384
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"

# name -> (ideal_dist, selection, episodes, "weak": per GPU | "strong": in total, BASELINE.json config it is)
WORKLOADS = {
    "episodes": ("3-20-10-weighted", "degree", 16384, "weak", "configs[1]"),
    "u3": ("3-20-10-uniform", "degree", 65536, "strong", "configs[2]"),
    "u5": ("5-5-10-uniform", "degree", 65536, "strong", "configs[2]"),
    "cyclic6": ("cyclic-6", "random", 1024, "weak", "configs[4]"),
}
SCALING, CONFIG_ID, DATA_NOTE = "weak", "configs[1]", ""
SEL_SEED = 1234  # Random selection: episode e draws choice() from minstd_rand0 seeded SEL_SEED + e


def workload_string():
    """config.workload: the same string in both arms (the driver compares them)."""
    return "%s, %d episodes %s to completion, %s selection (BASELINE %s)" % (
        DIST, EPISODES, "per GPU" if SCALING == "weak" else "in total, sharded", STRATEGY, CONFIG_ID)


def algorithmic_bytes(c):
    """SURVEY 8(d): 12 B per term read/written by an addition, 8 B per reducer lead monomial examined,
    24 B per lead term moved to the remainder, 8 B per basis / pair entry touched by update()."""
    return (12 * (c["terms_read"] + c["terms_written"]) + 8 * c["lms_scanned"] + 24 * c["term_moves"]
            + 8 * (c["update_basis"] + c["update_pairs"]))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_capture():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


def ncu_traffic(kernel):
    """DRAM bytes per launch of the workload's dominant kernel from a committed ncu --set full capture of the same
    command, or None when no capture of that kernel / workload is committed."""
    return ncu_capture().get(kernel + "_dram_bytes_per_launch")


def int_pipe(kernel, kernel_s, sm_mhz, sm_count, counters):
    """The secondary roofline BASELINE.json allows for this path (SURVEY 8(d)), both ways of counting it:
    `issue`: warp instructions per launch of the kernel (a property of kernel + workload, from the committed ncu
    capture of the same command) over the kernel's OWN live launch time, against SMs x 4 schedulers x SM clock;
    `algorithmic`: SURVEY 8(d)'s integer-op model -- 10 thread-int-ops per merged output term, 5 per reducer lead
    monomial examined -- against SMs x 4 sub-partitions x 16 INT32 lanes x SM clock."""
    if not sm_mhz or not kernel_s:
        return None
    c = ncu_capture()
    clk = sm_mhz * 1e6
    ops = 10.0 * counters["terms_written"] + 5.0 * counters["lms_scanned"]
    peak_ops = sm_count * 4 * 16 * clk
    out = {"kernel": kernel, "kernel_ms": kernel_s * 1e3, "sm_mhz": sm_mhz,
           "algorithmic": {"int_ops_per_launch": ops, "achieved": ops / kernel_s / 1e12, "peak": peak_ops / 1e12,
                           "unit": "T thread-int-op/s", "frac": ops / kernel_s / peak_ops,
                           "model": "10 per output term + 5 per lead monomial scanned (SURVEY 8(d)); peak = SMs x 4 x 16 x clock"}}
    inst = c.get(kernel + "_warp_instructions_per_launch")
    if inst:
        peak = sm_count * 4 * clk
        out["issue"] = {"achieved": inst / kernel_s / 1e9, "peak": peak / 1e9, "unit": "G warp-inst/s",
                        "frac": inst / kernel_s / peak, "warp_instructions_per_launch": inst,
                        "alu_pipe_pct_of_peak_while_active": c.get(kernel + "_alu_pipe_pct_active"),
                        "issue_slots_busy_pct": c.get(kernel + "_issue_active_pct"),
                        "threads_per_warp_instruction": c.get(kernel + "_threads_per_warp_instruction"),
                        "source": c.get(kernel + "_source") or c.get("source")}
    return out


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU every ~2 ms through NVML (in-process thread) while the timed
    region runs -- the region is tens of milliseconds, far below nvidia-smi's sampling period."""

    def __init__(self, torch_index):
        import threading
        self.samples, self.reasons, self.max_mhz, self.err = [], set(), None, None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(torch_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        except Exception as ex:  # no NVML: report that instead of inventing clocks
            self.err = repr(ex)

    def _loop(self):
        nv = self.nv
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                 ("hw_power_brake", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown))
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for n, bit in names:
                    if r & bit:
                        self.reasons.add(n)
            except Exception as ex:
                self.err = repr(ex)
                return
            time.sleep(0.002)

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.samples:
            sm = sorted(self.samples)
            out["sm_mhz"] = sm[len(sm) // 2]
        if self.err:
            out["error"] = self.err
        return out


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_cpu_oracle():
    from oracle import oracle as O
    if O.have_ref():
        return O.load_ref(), "reference"
    return O.load_port(), "port"


def cpu_sample(orc, kind, seconds, threads):
    """Times the reference env (reset + Degree select + step to completion) on `threads` host threads over a
    bounded sample of the SAME workload (episodes seed 0..count-1), sized for about `seconds` of wall time."""
    if kind != "reference":
        threads = 1  # the C restatement is single-threaded
    n0 = (64 if STRATEGY != "random" else 1) * threads
    probe = cpu_run(orc, kind, 0, n0, threads)
    rate = probe["steps"] / max(probe["seconds"], 1e-9)
    steps_per_ep = probe["steps"] / float(n0)
    count = int(min(EPISODES, max(n0, seconds * rate / steps_per_ep)))
    if count > EPISODES // 2:
        count = EPISODES  # the whole workload fits the budget: no sampling at all
    r = cpu_run(orc, kind, 0, count, threads)
    if count == EPISODES and r["seconds"] < seconds / 2:
        # the whole workload is quicker than the time budget: repeat it so the figure is not a 0.2 s measurement
        reps = int(min(64, max(1, seconds / max(r["seconds"], 1e-3)))) - 1
        for _ in range(reps):
            q = cpu_run(orc, kind, 0, count, threads)
            for k in ("steps", "additions", "seconds"):
                r[k] += q[k]
        r["reps"] = reps + 1
    return r, count, threads


def cpu_run(orc, kind, seed0, count, threads):
    """Episodes seed0 .. seed0+count-1 of the current workload on the host: the reference env stepped with the
    selection comparators (First/Degree/Normal/Sugar), or the reference's own buchberger() loop for seeded Random."""
    if STRATEGY == "random":
        if kind != "reference":
            raise SystemExit("the Random-selection CPU arm needs oracle/_ref (the unmodified reference)")
        return orc.bench_buchberger(DIST, STRATEGY, seed0, count, nthreads=threads, sel_seed0=SEL_SEED + seed0)
    return orc.bench_selection(DIST, STRATEGY, seed0, count, nthreads=threads)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    orc, kind = load_cpu_oracle()
    threads = host_threads()
    # each step = the first `count` episodes of the workload, sized for ~4 s per step
    probe, count, threads = cpu_sample(orc, kind, 4.0, threads)
    for _ in range(args.warmup):
        cpu_run(orc, kind, 0, max(count // 8, threads), threads)
    steps = adds = 0
    secs = 0.0
    for _ in range(args.steps):
        r = cpu_run(orc, kind, 0, count, threads)
        steps += r["steps"]; adds += r["additions"]; secs += r["seconds"]
    value = steps / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * secs / args.steps, "higher_is_better": True,
        "scaling": SCALING, "vs_baseline": None, "dtype": "int32 (GF(32003) coefficients, int exponent vectors)",
        "data": DATA_NOTE.replace("on-device restatement of the reference", "reference"),
        "config": {"workload": workload_string(), "sample": "bounded sample: episodes 0..%d of %d per step" % (count - 1, EPISODES),
                   "episodes_per_step": count, "host_threads": threads},
        "additions_per_sec": adds / secs,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "%d episodes (seeds 0..%d) x %d steps, one BuchbergerEnv per thread, "
                                   "env.seed(e); reset(); %s until P empty"
                                   % (count, count - 1, args.steps,
                                      "the reference buchberger() loop with seeded Random selection" if STRATEGY == "random"
                                      else STRATEGY + " select + step")},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


RECORD_FIELDS = ("steps", "additions", "zero_reductions", "nonzero_reductions", "nbasis", "nterms", "status", "rerolls",
                 "trace_hash", "basis_hash", "discounted_return")
GB_FIELDS = ("gb_hash", "gb_polys", "gb_terms")


def record_mismatches(orc, kind, runs, dist, selection, n, seed0, sel_seed0):
    """{"<name>.<field>": episodes} for every field in which the first n records of runs[name] = (records, fields)
    differ from the unmodified reference's records of the same episodes, and a description of what they were compared
    with: the reference itself on the host threads where oracle/_ref is built, else the stored digests of its records
    (tests/golden/records.json; the count of a differing field is then 1)."""
    bad = {}
    if kind == "reference":
        t0 = time.perf_counter()
        want = orc.run_records(dist, selection, n, seed0=seed0, sel_seed0=sel_seed0, gamma=0.99, compute_gb=True)
        for name, (got, fields) in runs.items():
            for f in fields:
                m = int((got[f][:n] != want[f]).sum())
                if m:
                    bad["%s.%s" % (name, f)] = m
        return bad, ("unmodified reference (oracle/_ref: BuchbergerEnv seed/reset/step + interreduce(minimalize(G)), "
                     "buchberger.cpp:299-329, 102-122), %.1f s on the host threads" % (time.perf_counter() - t0))
    from oracle import golden
    k = golden.key(dist, selection, n, seed0=seed0, sel_seed0=sel_seed0)
    if not golden.have(k):
        raise SystemExit("bench.py: the parity gate needs oracle/_ref (the unmodified reference compiled by oracle/Makefile) "
                         "or stored records of run %s (tests/golden/make_records.py)" % k)
    for name, (got, fields) in runs.items():
        for f in golden.mismatches(got[:n], k, fields):
            bad["%s.%s" % (name, f)] = 1
    return bad, "digests of the unmodified reference's records of run %s (tests/golden/records.json)" % k


def parity_gate(orc, kind, timed, with_gb, ep_first, limit):
    """Every episode record of the timed output (`timed`, compute_gb = 0) and of the extra launch with the reduced
    Groebner basis (`with_gb`) against the unmodified reference's records.  Returns the `parity` object; raises
    SystemExit on any mismatch (no value is printed then)."""
    n = len(timed) if not limit else min(limit, len(timed))
    runs = {"timed": (timed, RECORD_FIELDS), "with_gb": (with_gb, RECORD_FIELDS + GB_FIELDS)}
    bad, against = record_mismatches(orc, kind, runs, DIST, STRATEGY, n, ep_first, SEL_SEED + ep_first)
    mism = int(sum(bad.values()))
    out = {"episodes_checked": n, "episodes_in_launch": len(timed), "mismatches": mism,
           "fields": list(RECORD_FIELDS) + list(GB_FIELDS), "against": against}
    if mism:
        raise SystemExit("bench.py: PARITY FAILURE, no value reported: %r" % (bad,))
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays, dtype):
    """--dump-outputs: writes every array (one row per episode / environment) as <path>/<name>.npy in `dtype`, and the
    row indices as <path>/rows.npy.  Above 64 MiB in all, the same fixed, seeded sample of rows is taken of every array."""
    import numpy as np
    n = len(next(iter(arrays.values())))
    row_bytes = 8 + sum(np.dtype(dtype).itemsize * (a.size // max(n, 1)) for a in arrays.values())
    keep = min(n, (DUMP_BYTES - 128 * (len(arrays) + 1)) // row_bytes)   # 128 B: the header of a .npy file
    rows = np.arange(n) if keep >= n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a[rows]).astype(dtype))


def record_arrays(stats):
    """Episode records as arrays that float64 holds exactly: 64-bit checksums are split into 32-bit halves."""
    out = {}
    for f in stats.dtype.names:
        if stats[f].dtype.itemsize == 8 and stats[f].dtype.kind == "u":
            out[f + "_lo"], out[f + "_hi"] = stats[f] & 0xFFFFFFFF, stats[f] >> 32
        else:
            out[f] = stats[f]
    return out


def time_launches(torch, fn, steps, flush):
    """Device time of `steps` calls of fn(), L2 flushed before each: (total ms, [ms])."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.fill_(1)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    return sum(ms), ms


def extra_step_api(torch, dev, local, flush):
    """The step API that IS the drop-in for a vectorised trainer: per call one bb_select (Degree) + one bb_step_observe
    (step, auto-reset, state matrix of pmax = 64 rows, |P|, reward, done) for 16384 LeadMonomialsEnv(k=2) environments,
    16 calls captured in one CUDA graph.  env steps = environments x calls (auto-reset keeps every environment running)."""
    from deepgroebner_b200 import LeadMonomialsEnv
    N, PMAX, G = 16384, 64, 16
    env = LeadMonomialsEnv(DIST, k=2, num_envs=N, device="cuda:%d" % local, pmax=PMAX)
    eng = env.engine
    eng.seed(0)
    eng.set_auto_reset(True)
    eng.reset()
    acts = torch.empty(N, dtype=torch.int32, device=dev)
    obs = torch.empty((N, PMAX, eng.cols), dtype=torch.int32, device=dev)
    lens = torch.empty(N, dtype=torch.int32, device=dev)
    rew = torch.empty(N, dtype=torch.float64, device=dev)
    done = torch.empty(N, dtype=torch.uint8, device=dev)

    def one():
        eng.select(STRATEGY, out=acts)
        eng.step_observe(acts, PMAX, reward=rew, done=done, obs=obs, lengths=lens)

    for _ in range(8):
        one()
    torch.cuda.synchronize()
    eng.counters(reset=True)
    tot, _ = time_launches(torch, lambda: [one() for _ in range(G)], 5, flush)
    eager = N * G * 5 / (tot / 1e3)
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        one()
        torch.cuda.synchronize()
        with torch.cuda.graph(graph, stream=s):
            for _ in range(G):
                one()
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    eng.counters(reset=True)
    tot, _ = time_launches(torch, graph.replay, 10, flush)
    c = eng.counters(reset=True)
    assert c["env_steps"] == N * G * 10, (c["env_steps"], N * G * 10)
    return {"value": N * G * 10 / (tot / 1e3), "unit": UNIT, "eager_launches": eager, "environments": N, "pmax": PMAX,
            "calls_per_graph": G, "kernels_per_call": 3, "obs_bytes_per_call": int(obs.numel() * 4),
            "what": "bb_select(degree) + bb_step_observe (k_prefill: the environments' queues of prepared next episodes, topped up "
                    "every 32nd call; k_step_obs: step + auto-reset + state matrix + |P| + reward + done) per call, device-timed, "
                    "L2 flushed between graph replays"}


def extra_dropin_n1(seconds=2.0):
    """LeadMonomialsEnv(num_envs=1) driven exactly like the reference's scripts/random_episodes.py:30-41 drives
    CLeadMonomialsEnv (reset, uniform-random row, step until done), host call by host call -- the class INTEGRATION.md
    tells a maintainer to switch to -- beside the reference's own Cython binding timed on this box (oracle/_ref)."""
    import numpy as np
    from deepgroebner_b200 import LeadMonomialsEnv

    def drive(env, secs):
        rng = np.random.default_rng(0)
        n = eps = 0
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < secs:
            s = env.reset()
            done = False
            while not done:
                s, r, done, _ = env.step(int(rng.integers(len(s))))
                n += 1
            eps += 1
        return n / (time.perf_counter() - t0), eps

    env = LeadMonomialsEnv(DIST, k=2, num_envs=1, pmax=256)
    env.seed(0)
    drive(env, 0.3)
    ours, eps = drive(env, seconds)
    out = {"value": ours, "unit": UNIT, "episodes": eps,
           "what": "LeadMonomialsEnv(k=2, num_envs=1): reset()/step() answered by the handle's resident warp through a mailbox in "
                   "mapped host memory (bb_set_serve), state matrix returned as a numpy array (bb_reset_host / bb_step_host)"}
    env.engine.set_serve(False)
    drive(env, 0.2)
    out["launch_per_call"] = {"value": drive(env, seconds / 2)[0], "unit": UNIT,
                              "what": "the same with one kernel launch + a ticket in mapped host memory per call"}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        from deepgroebner_ref.wrapped import CLeadMonomialsEnv
        ref = CLeadMonomialsEnv(DIST, k=2)
        ref.seed(0)
        drive(ref, 0.2)
        r, _ = drive(ref, seconds)
        out["reference_cython"] = {"value": r, "unit": UNIT, "cores": 1,
                                   "what": "the reference's own CLeadMonomialsEnv (wrapped.pyx:11-38) built unmodified by "
                                           "oracle/build_cython_ref.sh, same loop, one host thread"}
    except Exception as ex:  # the Cython build does not exist on this box: say so instead of inventing a number
        out["reference_cython"] = {"unavailable": repr(ex)[:200]}
    return out


def extra_cyclic6(torch, local, orc, kind):
    """BASELINE configs[4] beside the headline: cyclic-6, seeded Random selection.  A launch lasts at least as long as its
    longest episode (697 000 dependent additions in the longest of 1024), so three figures: one launch of 1024 episodes
    alone; a pipeline of nine such launches on three alternating streams (the CTAs of the next batches move in while the longest
    episodes of the current one finish: the steady state of a job of many batches, as in the headline); one launch of
    8192 episodes.  The first 256 records of the 1024-episode launch are checked against the reference."""
    import numpy as np
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine("cyclic-6", num_envs=1024, device="cuda:%d" % local)
    out = {"what": "cyclic-6 over GF(32003), seeded Random selection (episode e: minstd_rand0 seeded %d + e), k_run_wide "
                   "(one CTA per environment, dividend as streams)" % SEL_SEED}
    dt = np.dtype(_lib.STATS_DTYPE)
    streams = [torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.Stream()]
    bufs = [torch.empty(1024 * 72, dtype=torch.uint8, device="cuda:%d" % local) for _ in streams]
    eng.run_episodes("random", episodes=64, selection_seed=SEL_SEED)
    for i in (1, 2):   # a stream's first call while the others are busy allocates its bank of environment slots
        with torch.cuda.stream(streams[i]):
            eng.run_episodes("random", episodes=64, selection_seed=SEL_SEED, to_host=False, out=bufs[i])
    torch.cuda.synchronize()

    peak, _ = measured_peak()

    def figures(ms, st, launches=1):
        adds, steps = int(st["additions"].sum()) * launches, int(st["steps"].sum()) * launches
        rate = adds / (ms / 1e3)
        # SURVEY 8(d): the reference's addition moves 3.8 KB on cyclic-6 (129 terms read, 127 written, 93 lead monomials
        # scanned, measured under Random selection); the stream reducer never materialises the dividend, so this is the
        # traffic of the algorithm it replaces at the rate it achieves, not bytes this kernel moves
        return {"ms": ms, "additions_per_sec": rate, "env_steps_per_sec": steps / (ms / 1e3), "additions": adds, "env_steps": steps,
                "hbm_equivalent": {"gbs": rate * 3800.0 / 1e9, "frac_of_peak": rate * 3800.0 / 1e9 / peak,
                                   "bytes_per_addition": 3800}}

    for n in (1024, 8192):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        buf, _ = eng.run_episodes("random", episodes=n, selection_seed=SEL_SEED, to_host=False)
        b.record()
        torch.cuda.synchronize()
        st = buf.cpu().numpy().view(dt)[:n].copy()
        assert (st["status"] == 2).all()
        out["episodes_%d" % n] = figures(a.elapsed_time(b), st)
        if n == 1024:
            st1024 = st
            bad, _ = record_mismatches(orc, kind, {"episodes_1024": (st, RECORD_FIELDS)}, "cyclic-6", "random", 256, 0, SEL_SEED)
            if bad:
                raise SystemExit("bench.py: PARITY FAILURE on cyclic-6: %r" % (bad,))
            out["parity"] = {"episodes_checked": 256, "mismatches": 0}
    L = 9
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(streams[0])
    for x in streams[1:]:
        x.wait_event(t0)
    for i in range(L):
        with torch.cuda.stream(streams[i % 3]):
            eng.run_episodes("random", episodes=1024, selection_seed=SEL_SEED, to_host=False, out=bufs[i % 3])
    for x in streams[1:]:
        streams[0].wait_stream(x)
    t1.record(streams[0])
    torch.cuda.synchronize()
    for bf in bufs:   # every batch of the pipeline produced the records of the single launch
        got = bf.cpu().numpy().view(dt)[:1024]
        assert all(np.array_equal(got[f], st1024[f]) for f in RECORD_FIELDS)
    out["episodes_1024_pipelined"] = dict(figures(t0.elapsed_time(t1), st1024, L), launches=L,
                                          what="nine launches of 1024 episodes on three alternating streams (three banks of "
                                               "environment slots), whole span")
    return out


def gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    from deepgroebner_b200 import sharding
    from deepgroebner_b200.ideals import FixedIdealGenerator, parse_ideal_dist
    spec = parse_ideal_dist(DIST, 32003)
    fixed = isinstance(spec, FixedIdealGenerator)
    nvars = spec.nvars() if fixed else spec.n
    if SCALING == "weak":   # every rank runs its own EPISODES episodes, disjoint seeds
        ep_first, ep_local = rank * EPISODES, EPISODES
    else:                   # EPISODES in total, contiguous blocks (deepgroebner_b200/sharding.py)
        ep_first, ep_local = sharding.shard_range(EPISODES, rank, world)
    slots = args.slots or min(resident_envs(local, nvars), ep_local)
    eng = BuchbergerEngine(DIST, num_envs=slots, device="cuda:%d" % local)
    eng.set_episode_offset(ep_first)   # selection seeds (and staged ideals) follow the global episode index
    kernel = "k_run_wide" if fixed else "k_run"
    seeds_host = torch.arange(ep_first, ep_first + ep_local, dtype=torch.int32).pin_memory()
    seeds_dev = seeds_host.to(dev)
    stats_bytes = ep_local * 72
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    main, alt, side = torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.Stream()
    runners = [main, alt]
    outs = [torch.empty(stats_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
    pipelined = ep_local <= 65536 and not args.no_pipeline

    def prepare(seeds):
        with torch.cuda.stream(side):
            return eng.prepare_episodes(ep_local, seeds=seeds)

    def run(seeds, gb=False, **kw):
        return eng.run_episodes(STRATEGY, episodes=ep_local, seeds=seeds, selection_seed=SEL_SEED, gamma=0.99,
                                compute_gb=gb, **kw)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def device_steps(n):
        """n steps.  Pipelined (the default): the runner of step i goes to stream i % 2, so the CTAs of batch i + 1 move in
        while batch i drains (an episode runner ends with its longest episodes on a mostly idle GPU), and the preparation
        runs two batches ahead on a third stream; the L2 flush write of a step sits on that step's stream in front of its
        runner.  The timed span is first event -> everything finished, divided by n.  Otherwise: one stream, prepare then
        run, L2 flushed between steps outside the event pairs.  Returns (ms, per-step event pairs, last output buffer)."""
        ev = []
        torch.cuda.synchronize()
        if not pipelined:
            for i in range(n):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                buf, _ = run(seeds_dev, to_host=False, out=outs[0])
                b.record()
                ev.append((a, b))
            torch.cuda.synchronize()
            return sum(a.elapsed_time(b) for a, b in ev), ev, buf, eng.counters(reset=True)
        prepare(seeds_dev)            # batches 0 and 1 (K preparations lie inside the span: those of batches 2 .. K + 1)
        prepare(seeds_dev)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(main)
        alt.wait_event(t0)
        side.wait_event(t0)
        for i in range(n):
            with torch.cuda.stream(runners[i % 2]):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                buf, _ = run(seeds_dev, to_host=False, out=outs[i % 2])
                b.record()
                ev.append((a, b))
            prepare(seeds_dev)
        main.wait_stream(alt)
        main.wait_stream(side)
        t1.record(main)
        torch.cuda.synchronize()
        c = eng.counters(reset=True)
        for _ in range(2):   # the two batches prepared ahead at the end of the span: run them off (untimed)
            run(seeds_dev, to_host=False)
        torch.cuda.synchronize()
        eng.counters(reset=True)
        return t0.elapsed_time(t1), ev, buf, c

    device_steps(max(args.warmup, 3))
    barrier()
    eng.counters(reset=True)

    # ---- device-timed region: K steps
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    wall0 = time.perf_counter()
    dev_ms, ev, buf, counters = device_steps(args.steps)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if sampler else None
    stats = buf.cpu().numpy().view(np.dtype(_lib.STATS_DTYPE))[:ep_local].copy()
    assert (stats["status"] == 2).all(), "not every episode finished: status histogram %r" % (
        dict(zip(*[x.tolist() for x in np.unique(stats["status"], return_counts=True)])),)
    steps_per_launch = int(stats["steps"].sum())
    adds_per_launch = int(stats["additions"].sum())
    assert counters["env_steps"] == steps_per_launch * args.steps

    # ---- end to end through the public API with host buffers.  Per step: pinned seeds H2D (with the preparation, two
    # batches ahead), runner, episode records D2H into pinned memory; the host waits for and reads the records of step
    # i - 1 while step i is in flight.
    host_out = [torch.empty(stats_bytes, dtype=torch.uint8).pin_memory() for _ in range(2)]

    def e2e_steps(n):
        """Seconds of n end-to-end steps (host clock, barrier on both sides) and the env steps the host read back."""
        barrier()
        t0 = time.perf_counter()
        seen = 0
        if pipelined:
            ahead = [prepare(seeds_host), prepare(seeds_host)]
            done = []
            for i in range(n):
                with torch.cuda.stream(runners[i % 2]):
                    b_, _ = run(ahead[i], to_host=False, out=outs[i % 2])
                    host_out[i % 2].copy_(b_, non_blocking=True)
                    e_ = torch.cuda.Event()
                    e_.record()
                    done.append(e_)
                ahead.append(prepare(seeds_host))
                if i >= 1:
                    done[i - 1].synchronize()
                    seen += int(host_out[(i - 1) % 2].numpy().view(np.dtype(_lib.STATS_DTYPE))["steps"][:ep_local].sum())
            done[-1].synchronize()
            seen += int(host_out[(n - 1) % 2].numpy().view(np.dtype(_lib.STATS_DTYPE))["steps"][:ep_local].sum())
            barrier()
            secs = time.perf_counter() - t0
            for _ in range(2):   # run off the batches prepared ahead (untimed)
                run(seeds_dev, to_host=False)
            torch.cuda.synchronize()
        else:
            for _ in range(n):
                st_, _ = run(seeds_host, out_host=host_out[0])
                seen += int(st_["steps"].sum())
            barrier()
            secs = time.perf_counter() - t0
        return secs, seen

    e2e_steps(3)   # first use allocates the seed ring and pins nothing new afterwards
    e2e_s, seen = e2e_steps(args.steps)
    assert seen == steps_per_launch * args.steps, (seen, steps_per_launch * args.steps)
    eng.counters(reset=True)

    # ---- the kernels on their own (outside the timed regions): unpipelined launches with events inside bb_run
    eng.set_timing(True)
    kprep, krun = [], []
    for _ in range(5):
        flush.fill_(1)
        run(seeds_dev, to_host=False)
        p_ms, r_ms = eng.last_run_ms()
        kprep.append(p_ms); krun.append(r_ms)
    eng.set_timing(False)
    kernel_counters = eng.counters(reset=True)
    kprep_ms, krun_ms = float(np.median(kprep)), float(np.median(krun))

    # ---- one launch with the reduced Groebner basis (outside the timed regions), timed for `with_gb`
    gb_tot, _ = time_launches(torch, lambda: run(seeds_dev, gb=True, to_host=False), 3, flush)
    gb_buf, _ = run(seeds_dev, gb=True, to_host=False)
    gb_stats = gb_buf.cpu().numpy().view(np.dtype(_lib.STATS_DTYPE))[:ep_local].copy()
    eng.counters(reset=True)

    # ---- parity gate: every rank checks every episode of its own shard
    orc, kind = load_cpu_oracle()
    limit = args.parity_episodes or (1024 if fixed else 0)
    parity = parity_gate(orc, kind, stats, gb_stats, ep_first, limit)

    t = torch.tensor([dev_ms, e2e_s * 1000.0], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(steps_per_launch), float(adds_per_launch), float(parity["episodes_checked"]),
                        float(parity["mismatches"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max = float(t[0]), float(t[1])
    total_steps, total_adds = float(tot[0]), float(tot[1])
    parity["episodes_checked"], parity["mismatches"] = int(tot[2]), int(tot[3])
    per_rank = None
    if world > 1:   # diagnosis of the scaling figure: every rank's own device time, fastest single launch and work
        mine = torch.tensor([dev_ms / args.steps, min(a.elapsed_time(b) for a, b in ev), float(steps_per_launch)],
                            dtype=torch.float64, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_step": [round(float(x[0]), 4) for x in allr], "min_ms": [round(float(x[1]), 4) for x in allr],
                    "env_steps_per_launch": [int(x[2]) for x in allr]}

    if rank == 0:
        peak, peak_src = measured_peak()
        per_launch = {k: v / 5.0 for k, v in kernel_counters.items()}   # the 5 unpipelined launches above
        abytes = algorithmic_bytes(per_launch)
        kernel_s = krun_ms / 1000.0
        achieved = abytes / kernel_s / 1e9
        value = total_steps * args.steps / (dev_ms_max / 1000.0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": SCALING, "vs_baseline": None,
            "dtype": "u64 packed monomials + u32 GF(32003) coefficients (integer)",
            "data": DATA_NOTE,
            "config": {"workload": workload_string(),
                       "episodes_per_gpu": ep_local, "env_steps_per_launch": steps_per_launch, "slots": slots,
                       "parallelism": "episodes sharded across GPUs, no collective on the step path",
                       "pipeline": ("steps are pipelined like the batches of one job: the runner of step i on stream i % 2 (the CTAs "
                                    "of batch i + 1 move in while batch i drains), preparation (k_prepare_lanes + k_order) two "
                                    "batches ahead on a third stream; timed span = first event to all streams idle, / steps")
                                   if pipelined else "none: prepare, then run, on one stream; sum of the steps' event pairs",
                       "l2": "160 MiB flush write (L2: 126 MB) in front of every step's runner" + (" (inside the timed span)" if pipelined else "")},
            "additions_per_sec": total_adds * args.steps / (dev_ms_max / 1000.0),
            "spair_reductions_per_sec": value,
            # per step: k_prepare(_lanes) + k_order + the runner (one batch) -- the L2 flush fill and the queue memset are not ours
            "gpu_launches": 3 * args.steps * ((ep_local + 65535) // 65536),
            "wall_s_timed_region": wall,
            "step_ms": [round(a.elapsed_time(b), 4) for a, b in ev],
            "clocks": clocks,
            "parity": parity,
            "e2e": {"value": total_steps * args.steps / (e2e_ms_max / 1000.0), "unit": UNIT,
                    "h2d_bytes_per_step": ep_local * 4, "d2h_bytes_per_step": stats_bytes,
                    "api": "BuchbergerEngine.prepare_episodes(seeds=pinned host) + run_episodes + records copied to pinned host "
                           "memory and read by the host, one step behind the step in flight"},
            "kernel_ms": {"prepare+order": kprep_ms, kernel: krun_ms,
                          "how": "CUDA events inside bb_run (bb_set_timing), median of 5 unpipelined launches, L2 flushed"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(kernel) if args.workload == "episodes" or fixed else None,
                         "peak_source": peak_src, "kernel": kernel, "kernel_ms": krun_ms,
                         "algorithmic_bytes_per_launch": abytes,
                         "note": ("terms_read / terms_written count the reducers only: the dividend is never materialised "
                                  "(bb_streams.cuh)") if fixed else
                                 "latency/integer bound at binomial sizes (working set lives in L1/L2); see DESIGN.md"},
            "with_gb": {"value": steps_per_launch * 3 / (gb_tot / 1000.0), "unit": UNIT, "n_gpus": 1,
                        "what": "the same launch with compute_gb = 1 (interreduce(minimalize(G)) + checksum per episode), "
                                "rank 0, unpipelined, 3 launches"},
            "counters_per_launch": per_launch,
        }
        if per_rank:
            line["per_rank"] = per_rank
        ip = int_pipe(kernel, kernel_s, (clocks or {}).get("sm_mhz"), eng.sm_count, per_launch)
        if ip:
            line["int_pipe"] = ip
        if world == 1 and not args.no_cpu:
            threads = host_threads()
            r, count, threads = cpu_sample(orc, kind, args.cpu_seconds, threads)
            line["cpu_baseline"] = {
                "value": r["steps"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": kind,
                "sample": "%d episodes (seeds 0..%d) of the same workload x %d passes, one reference BuchbergerEnv per "
                          "host thread, %.1f s" % (count, count - 1, r.get("reps", 1), r["seconds"])}
        if world == 1 and not args.no_extras and args.workload == "episodes":
            del eng
            torch.cuda.empty_cache()
            line["step_api"] = extra_step_api(torch, dev, local, flush)
            line["dropin_n1"] = extra_dropin_n1()
            line["cyclic6"] = extra_cyclic6(torch, local, orc, kind)
        if args.dump_outputs:   # the records of the last timed step
            dump_outputs(args.dump_outputs, record_arrays(stats), "float64")
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def rollout_arm(args):
    """BASELINE configs[3]: LeadMonomialsEnv(k=2) PPO rollout -- env step + PMLP(128) policy head sampling on device,
    fused in one launch (bb_rollout), auto-reset.  Extra workload (`--workload rollout`); the default stays configs[1]."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from deepgroebner_b200 import LeadMonomialsEnv
    from deepgroebner_b200.rollout import PairsPolicy

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    N, T = args.envs, args.horizon
    env = LeadMonomialsEnv(DIST, k=2, num_envs=N, device="cuda:%d" % local, pmax=64)
    env.seed(np.arange(rank * N, rank * N + N))
    env.engine.set_auto_reset(True)
    env.engine.reset()
    net = PairsPolicy(env.engine.cols, 128, torch_seed=0, seed=1, device=dev)
    out = env.engine.rollout(net, T)
    host = {k: torch.empty_like(out[k], device="cpu").pin_memory() for k in ("reward", "done")}
    w_host = [t.cpu().pin_memory() for t in net.parameters()]
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for i in range(max(args.warmup, 3)):
        flush.fill_(1)
        env.engine.rollout(net, T, counter0=i * T, out=out)
    torch.cuda.synchronize()
    env.engine.counters(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i, (a, b) in enumerate(ev):
        flush.fill_(1)
        a.record()
        env.engine.rollout(net, T, counter0=(100 + i) * T, out=out)
        b.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    last = {k: v.cpu().numpy() for k, v in out.items()} if args.dump_outputs and rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    counters = env.engine.counters(reset=True)
    steps_done = counters["env_steps"]
    # end to end: weights from pinned host memory, rewards + done flags back to the host
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        for t, h in zip(net.parameters(), w_host):
            t.copy_(h, non_blocking=True)
        env.engine.rollout(net, T, counter0=(200 + i) * T, out=out)
        for k in host:
            host[k].copy_(out[k], non_blocking=True)
        torch.cuda.synchronize()
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_steps = env.engine.counters(reset=True)["env_steps"]
    t = torch.tensor([dev_ms, e2e_s * 1000.0], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(steps_done), float(e2e_steps)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank == 0:
        peak, peak_src = measured_peak()
        abytes = (algorithmic_bytes(counters) + 4 * 12 * counters["obs_rows"]) / args.steps
        achieved = abytes / (dev_ms / 1000.0 / args.steps) / 1e9
        line = {
            "metric": "rollout_env_steps_per_sec", "value": float(tot[0]) / (float(t[0]) / 1000.0), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": float(t[0]) / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 packed monomials + u32 GF(32003) coefficients (integer); fp32 policy head",
            "data": "synthetic (device generator, env e = stream seed e; PMLP(128) Glorot-initialised, torch seed 0)",
            "config": {"workload": "%s LeadMonomialsEnv(k=2), %d envs x %d fused steps per launch, PMLP(128) sampling on "
                                   "device, auto-reset (BASELINE configs[3])" % (DIST, N, T),
                       "envs_per_gpu": N, "horizon": T, "l2": "160 MiB flush write (L2: 126 MB) between timed launches"},
            "gpu_launches": args.steps, "clocks": clocks,   # one fused k_rollout per step
            "e2e": {"value": float(tot[1]) / (float(t[1]) / 1000.0), "unit": UNIT,
                    "h2d_bytes_per_step": sum(x.numel() * 4 for x in w_host),
                    "d2h_bytes_per_step": sum(h.numel() * h.element_size() for h in host.values())},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "kernel": "k_rollout",
                         "algorithmic_bytes_per_launch": abytes},
        }
        if world == 1 and not args.no_cpu:
            orc, kind = load_cpu_oracle()
            if kind == "reference":
                threads = host_threads()
                r = orc.bench_random(DIST, 0, 2000 * threads, nthreads=threads)
                line["cpu_baseline"] = {"value": r["steps"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": kind,
                                        "sample": "scripts/random_episodes.cpp loop (uniform-random actions, no network) on "
                                                  "LeadMonomialsEnv(k=2), %d episodes, %.1f s" % (2000 * threads, r["seconds"])}
        if last is not None:   # what the last timed launch returned
            dump_outputs(args.dump_outputs, last, "float32")
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default=os.environ.get("BB_BENCH_WORKLOAD", "episodes"), choices=sorted(WORKLOADS) + ["rollout"],
                    help="episodes = BASELINE configs[1] (the headline); u3/u5 = configs[2]; cyclic6 = configs[4]; "
                         "rollout = configs[3]")
    ap.add_argument("--episodes", type=int, default=0, help="override the workload's episode count")
    ap.add_argument("--envs", type=int, default=16384, help="rollout workload: environments per GPU")
    ap.add_argument("--horizon", type=int, default=128, help="rollout workload: fused steps per launch")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--slots", type=int, default=0, help="environment slots (0 = one resident wave)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the step_api / dropin_n1 / cyclic6 sub-objects")
    ap.add_argument("--no-pipeline", action="store_true", help="prepare every batch on the runner's stream (A/B)")
    ap.add_argument("--parity-episodes", type=int, default=0,
                    help="episodes of the launch checked against the reference (0 = all; cyclic-6: 1024)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy: the episode records, or the "
                         "rollout's arrays")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global DIST, STRATEGY, EPISODES, SCALING, CONFIG_ID, DATA_NOTE
    DIST, STRATEGY, EPISODES, SCALING, CONFIG_ID = WORKLOADS.get(args.workload, WORKLOADS["episodes"])
    if args.episodes:
        EPISODES = args.episodes
    DATA_NOTE = ("synthetic (fixed ideal staged on device; episode e = Random-selection stream seed %d + e)" % SEL_SEED
                 if STRATEGY == "random" else
                 "synthetic (on-device restatement of the reference RandomBinomialIdealGenerator; episode e = stream seed e)")
    if args.impl == "reference":
        reference_arm(args)
    elif args.workload == "rollout":
        rollout_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
