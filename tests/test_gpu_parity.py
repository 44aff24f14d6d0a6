"""GPU parity tests: the CUDA path (through the C-ABI / Python env classes) against the oracle and the golden
fixtures recorded from the unmodified reference.  Bit-exact: pair sequence, per-step reward, episode length,
basis, final reduced Groebner basis, observation matrices."""
import numpy as np
import pytest

from hashing import polys_hash, trace_hash
from helpers import episode_id, expand, golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def best_oracle():
    from oracle import oracle as O
    return O.load_ref() if O.have_ref() else O.load_port()


def trim(F, n=8):
    return [[(c, tuple(e)[:n]) for c, e in f] for f in F]


EPISODES = golden()["episodes"]


@pytest.mark.parametrize("rec", EPISODES, ids=[episode_id(r) for r in EPISODES])
def test_step_api_replays_golden_episode(torch_cuda, rec):
    """reset()/select()/step() one call at a time, against episodes recorded from the unmodified reference."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from deepgroebner_b200.ideals import FixedIdealGenerator
    n = rec["nvars"]
    ideal = trim(expand(rec["ideal"]), n)
    kw = dict(elimination=rec["elimination"], rewards=rec["rewards"], sort_input=rec["sort_input"],
              sort_reducers=rec["sort_reducers"], k=1, num_envs=1)
    eng = BuchbergerEngine(rec["dist"], **kw)   # every recorded distribution is drawn by the device generator
    eng.seed(rec["seed"])
    eng.reset()
    assert eng.basis(0) == ideal
    pairs, lengths = eng.pairs(eng.caps["max_pairs"])
    assert pairs[0, :int(lengths[0])].cpu().tolist() == rec["pairs0"]
    trace = []
    for t, row in enumerate(rec["trace"]):
        if "selection" in rec:
            a = eng.select(rec["selection"])
        else:
            a = torch_cuda.tensor([rec["actions"][t]], dtype=torch_cuda.int32, device="cuda")
        pairs, lengths = eng.pairs(eng.caps["max_pairs"])
        i, j = pairs[0, int(a[0])].cpu().tolist()
        reward, done = eng.step(a)
        st = eng.stats()[0]
        adds = int(-reward.item()) if rec["rewards"] == "additions" else row[2]
        if rec["rewards"] == "reductions":
            assert reward.item() == -1.0
        trace.append([i, j, adds, int(eng.lengths()[0]), int(st["nbasis"])])
        assert trace[-1] == row, "step %d" % t
        assert bool(done.item()) == (row[3] == 0)
    assert int(eng.status()[0]) == 2
    basis = eng.basis(0)
    assert [len(g) for g in basis] == rec["basis_len"]
    assert basis[-3:] == trim(expand(rec["last_basis"]), n)
    assert eng.final_gb(0) == trim(expand(rec["final_gb"]), n)
    st = eng.stats()[0]
    assert st["steps"] == len(rec["trace"])
    if rec["rewards"] == "additions":
        assert st["additions"] == sum(r[2] for r in rec["trace"])
        assert int(st["trace_hash"]) == trace_hash(np.array(rec["trace"]))


@pytest.mark.parametrize("rec", golden()["lm"], ids=lambda r: "%s-k%d" % (r["dist"], r["k"]))
def test_lead_monomials_env_matrices(torch_cuda, rec):
    """LeadMonomialsEnv(num_envs=1) returns exactly what wrapped.pyx returned for the reference."""
    from deepgroebner_b200 import LeadMonomialsEnv
    env = LeadMonomialsEnv(rec["dist"], k=rec["k"])
    env.seed(rec["seed"])
    s = env.reset()
    assert s.dtype == np.int32 and s.tolist() == rec["states"][0]
    for a, r, exp in zip(rec["actions"], rec["rewards"], rec["states"][1:]):
        s, reward, done, info = env.step(a)
        assert reward == r and s.tolist() == exp and done == (len(exp) == 0) and info == {}


@pytest.mark.parametrize("dist,strategy,episodes", [
    ("3-20-10-weighted", "degree", 1024), ("3-20-10-weighted", "first", 512), ("3-20-10-weighted", "normal", 512),
    ("3-20-10-uniform", "degree", 256), ("5-5-10-uniform", "degree", 256), ("5-5-10-uniform", "normal", 128),
    ("4-6-8-maximum-homog", "first", 128), ("3-12-6-weighted-pure", "normal", 128), ("2-9-5-uniform-consts", "degree", 128),
    # RandomIdealGenerator (Poisson-length polynomials, ideals.cpp:204-231) drawn on device
    ("3-6-5-0.5-uniform", "degree", 128), ("4-4-4-1.5-weighted-homog", "normal", 64), ("2-8-6-3.0-maximum-consts", "first", 64),
    ("3-5-4-0.5-weighted", "sugar", 64),
])
def test_run_episodes_bit_exact_vs_oracle(torch_cuda, dist, strategy, episodes):
    """bb_run (persistent kernel, on-device generator + selection): every episode's pair sequence, rewards, length,
    final basis and reduced GB equal the oracle's, via full traces for the first 32 and checksums for all."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    eng = BuchbergerEngine(dist, num_envs=min(episodes, 512))
    stats, trace = eng.run_episodes(strategy, episodes=episodes, seed_base=1000, compute_gb=True, trace_episodes=32,
                                    trace_cap=1024)
    env = orc.env(dist)
    for e in range(episodes):
        env.seed(1000 + e)
        env.reset()
        t = env.run(selection=strategy)
        s = stats[e]
        assert s["status"] == 2
        assert s["steps"] == len(t) and s["additions"] == int(t[:, 2].sum()), (e, s, len(t))
        assert s["nbasis"] == int(t[-1, 4]) if len(t) else True
        assert int(s["trace_hash"]) == trace_hash(t), e
        assert int(s["basis_hash"]) == polys_hash(env.basis()), e
        gb = env.final_gb()
        assert (s["gb_polys"], s["gb_terms"]) == (len(gb), sum(len(g) for g in gb))
        assert int(s["gb_hash"]) == polys_hash(gb), e
        if e < 32:
            assert np.array_equal(trace[e, :len(t)], t[:, :4]) and (trace[e, len(t):] == -1).all()
    c = eng.counters()
    assert c["env_steps"] == int(stats["steps"].sum()) and c["additions"] == int(stats["additions"].sum())
    assert c["episodes"] == episodes


def test_batched_step_matches_single_env_oracle(torch_cuda):
    """N=256 environments stepped together with per-env random actions == 256 independent oracle envs."""
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    N, k = 256, 2
    env = LeadMonomialsEnv("3-20-10-weighted", k=k, num_envs=N, pmax=256)
    env.seed(np.arange(500, 500 + N))
    refs = []
    for e in range(N):
        r = orc.lm_env("3-20-10-weighted", k=k)
        r.seed(500 + e)
        refs.append(r)
    obs, lengths = env.reset()
    states = [r.reset() for r in refs]
    rng = np.random.default_rng(3)
    for step in range(40):
        lens = lengths.cpu().numpy()
        o = obs.cpu().numpy()
        for e in range(N):
            assert lens[e] == len(states[e])
            assert np.array_equal(o[e, :lens[e]], states[e]) and (o[e, lens[e]:] == -1).all()
        acts = np.array([rng.integers(l) if l else 0 for l in lens], dtype=np.int32)
        (obs, lengths), reward, done, _ = env.step(torch.as_tensor(acts, device="cuda"))
        rw, dn = reward.cpu().numpy(), done.cpu().numpy()
        for e in range(N):
            if lens[e] == 0:
                assert rw[e] == 0.0 and dn[e]
                continue
            s, r, d, _ = refs[e].step(int(acts[e]))
            states[e] = s
            assert rw[e] == r and bool(dn[e]) == d


def test_buchberger_env_state_and_pair_actions(torch_cuda):
    """BuchbergerEnv(num_envs=1): state (G, P) and (i, j) actions as in buchberger.py:243-394."""
    from deepgroebner_b200 import BuchbergerEnv
    orc = best_oracle()
    env = BuchbergerEnv("3-20-10-uniform")
    ref = orc.env("3-20-10-uniform")
    env.seed(123)
    ref.seed(123)
    G, P = env.reset()
    G2, P2 = ref.reset()
    assert G == trim(G2, 3) and P == P2
    for pick in (3, 0, 5, 1):
        a = P[pick]
        (G, P), reward, done, _ = env.step(a)
        r2, d2 = ref.step(a)
        assert reward == r2 and done == d2
        assert G == trim(ref.basis(), 3) and P == ref.pairs()
    with pytest.raises(ValueError):
        env.step((0, 0))


def test_fixed_ideals_cyclic_and_bad_action(torch_cuda):
    torch = torch_cuda
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    for name, n in (("cyclic-4", 4), ("cyclic-5", 5)):
        eng = BuchbergerEngine(name, num_envs=4)
        stats, trace = eng.run_episodes("normal", episodes=4, compute_gb=True, trace_episodes=4, trace_cap=2048)
        env = orc.env(name)
        env.reset()
        t = env.run(selection="normal")
        for e in range(4):
            assert stats["steps"][e] == len(t) and np.array_equal(trace[e, :len(t)], t[:, :4])
            assert int(stats["gb_hash"][e]) == polys_hash(env.final_gb())
        assert eng.final_gb(0) == trim(env.final_gb(), n)
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=2)
    eng.seed(0)
    eng.reset()
    reward, done = eng.step(torch.tensor([10000, 0], dtype=torch.int32, device="cuda"))
    assert eng.status().cpu().tolist()[0] == 3 and bool(done[0]) and reward[0].item() == 0.0
    assert eng.status().cpu().tolist()[1] in (1, 2)


def test_exponent_overflow_is_flagged_not_wrapped(torch_cuda):
    """n=8 packs 6 value bits per exponent: x^40 * ... must raise OVERFLOW_EXPONENT instead of wrapping."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from deepgroebner_b200.ideals import FixedIdealGenerator
    e = lambda *v: tuple(v) + (0,) * (8 - len(v))
    F = [[(1, e(40, 40, 40, 0, 0, 0, 0, 1)), (1, e())], [(1, e(0, 0, 0, 40, 40, 0, 0, 1)), (1, e())]]
    eng = BuchbergerEngine(FixedIdealGenerator(F, 8), num_envs=1)
    stats, _ = eng.run_episodes("first", episodes=1)
    assert stats["status"][0] == 7


RECORD_FIELDS = ("steps", "additions", "zero_reductions", "nonzero_reductions", "nbasis", "nterms", "status", "rerolls",
                 "trace_hash", "basis_hash", "gb_hash", "gb_polys", "gb_terms", "discounted_return")


def assert_records_equal(got, want, what):
    """Every field of every episode record (bb_episode_stats) bit-equal: pair sequence + rewards (trace_hash), length,
    final basis, reduced Groebner basis, discounted return.  `want` is a records array or, from reference_records, the
    name of a run whose stored digests stand for the reference's records."""
    if isinstance(want, str):
        from oracle import golden
        bad = golden.mismatches(got, want, RECORD_FIELDS)
        assert not bad, "%s: %s differ from the reference's records (tests/golden/records.json)" % (what, bad)
        return
    assert len(got) == len(want)
    for f in RECORD_FIELDS:
        bad = np.nonzero(got[f] != want[f])[0]
        assert len(bad) == 0, "%s: %d episodes differ in %s, first %d: gpu %r reference %r" % (
            what, len(bad), f, bad[0], got[f][bad[0]], want[f][bad[0]])


def reference_records(dist, selection, count, seed0=0, sel_seed0=0, max_steps=0, **env_kw):
    """The unmodified reference's records of a run (gamma 0.99, reduced basis computed): run live on oracle/_ref where
    it is built, else the name of the run in tests/golden/records.json, for assert_records_equal."""
    from oracle import golden
    from oracle import oracle as O
    if O.have_ref():
        return O.load_ref().run_records(dist, selection, count, seed0=seed0, sel_seed0=sel_seed0, max_steps=max_steps,
                                        gamma=0.99, compute_gb=True, **env_kw)
    k = golden.key(dist, selection, count, seed0=seed0, sel_seed0=sel_seed0, max_steps=max_steps, **env_kw)
    assert golden.have(k), "no stored records of run %s: add it to tests/golden/make_records.py" % k
    return k


@pytest.mark.parametrize("strategy", ["degree", "first", "normal"])
def test_full_size_every_episode_16384(torch_cuda, strategy):
    """BASELINE configs[1] at full size: ALL 16384 episodes of 3-20-10-weighted under Degree / First / Normal, every
    record field against the unmodified reference env (buchberger.cpp:299-329 driven by oracle/ref_shim.cpp
    ref_run_records); plus counter identities and a bit-identical second run."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=3552)
    eng.counters(reset=True)
    s1, _ = eng.run_episodes(strategy, episodes=16384, seed_base=0, compute_gb=True)
    c = eng.counters(reset=True)
    s2, _ = eng.run_episodes(strategy, episodes=16384, seed_base=0, compute_gb=True)
    assert (s1["status"] == 2).all()
    assert c["episodes"] == 16384 and c["env_steps"] == int(s1["steps"].sum())
    assert c["additions"] == int(s1["additions"].sum())
    assert c["zero_reductions"] + c["nonzero_reductions"] == c["env_steps"]
    for f in RECORD_FIELDS:
        assert np.array_equal(s1[f], s2[f]), f
    assert (s1["additions"] >= s1["steps"]).all() and (s1["nbasis"] == 10 + s1["nonzero_reductions"]).all()
    assert_records_equal(s1, reference_records("3-20-10-weighted", strategy, 16384), "3-20-10-weighted/" + strategy)


@pytest.mark.parametrize("dist,s", [("3-20-10-uniform", 10), ("5-5-10-uniform", 10)])
def test_full_size_every_episode_65536(torch_cuda, dist, s):
    """BASELINE configs[2] at full size: ALL 65536 episodes of the uniform distributions under Degree selection (one
    resident wave of slots, like bench.py), every record field against the unmodified reference env."""
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    E = 65536
    eng = BuchbergerEngine(dist, num_envs=resident_envs(0, int(dist.split("-")[0])))
    eng.counters(reset=True)
    s1, _ = eng.run_episodes("degree", episodes=E, seed_base=0, compute_gb=True)
    c = eng.counters(reset=True)
    assert (s1["status"] == 2).all()
    assert c["episodes"] == E and c["env_steps"] == int(s1["steps"].sum()) and c["additions"] == int(s1["additions"].sum())
    assert c["zero_reductions"] + c["nonzero_reductions"] == c["env_steps"]
    assert (s1["additions"] >= s1["steps"]).all() and (s1["nbasis"] == s + s1["nonzero_reductions"]).all()
    assert_records_equal(s1, reference_records(dist, "degree", E), dist)


ALL_STRATEGIES = ["first", "degree", "normal", "sugar", "random", "last", "codegree", "strange", "spice"]


def test_run_beyond_one_batch_of_65536(torch_cuda):
    """bb_run splits a call into batches of 65536 episodes (staging arena, queue and order are reused, episode ids carry
    on): 70000 episodes with explicit seeds give, episode by episode, what two separate calls over the same seeds give,
    and a sample on both sides of the boundary equals the oracle."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    E, cut = 70000, 65536
    seeds = (np.arange(E, dtype=np.int64) * 7 + 3).astype(np.int32)
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=2048)
    whole, _ = eng.run_episodes("degree", episodes=E, seeds=seeds)
    head, _ = eng.run_episodes("degree", episodes=cut, seeds=seeds[:cut])
    tail, _ = eng.run_episodes("degree", episodes=E - cut, seeds=seeds[cut:])
    assert (whole["status"] == 2).all()
    for f in ("steps", "additions", "trace_hash", "basis_hash", "nbasis", "rerolls", "discounted_return"):
        assert np.array_equal(whole[f][:cut], head[f]) and np.array_equal(whole[f][cut:], tail[f]), f
    env = orc.env("3-20-10-weighted")
    for e in list(range(cut - 8, cut + 8)) + [0, E - 1]:
        env.seed(int(seeds[e]))
        env.reset()
        t = env.run(selection="degree")
        assert whole["steps"][e] == len(t) and int(whole["trace_hash"][e]) == trace_hash(t), e


@pytest.mark.parametrize("dist", ["3-20-10-weighted", "5-5-10-uniform"])
@pytest.mark.parametrize("strategy", ALL_STRATEGIES)
def test_all_selection_types_whole_episodes(torch_cuda, dist, strategy):
    """bb_run under every SelectionType (buchberger.h:111) == buchberger(F, selection, ..., seed) of the reference:
    reduction counts, additions, the discounted return (a gamma-weighted checksum of the reward sequence, exact in
    double) and the reduced Groebner basis; for the deterministic strategies also the full pair sequence."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    port = __import__("oracle.oracle", fromlist=["x"]).load_port()
    episodes, sel_seed = 48, 77
    # the reversed strategies build much larger bases than the default binomial preset holds
    big = dict(max_basis=4096, max_pairs=32768, max_terms=12288) if strategy in ("last", "codegree", "strange", "spice") else {}
    eng = BuchbergerEngine(dist, num_envs=episodes, **big)
    stats, trace = eng.run_episodes(strategy, episodes=episodes, seed_base=300, compute_gb=True, trace_episodes=episodes,
                                    trace_cap=2048, selection_seed=sel_seed, gamma=0.99)
    gen = orc.generator(dist)
    penv = port.env(dist)
    for e in range(episodes):
        env = orc.env(dist)
        env.seed(300 + e)
        F, _ = env.reset()     # the ideal the environment settled on (re-rolls included)
        gb, st = orc.buchberger(F, selection=strategy, gamma=0.99, seed=sel_seed + e)
        s = stats[e]
        assert s["status"] == 2
        assert (s["zero_reductions"], s["nonzero_reductions"], s["additions"]) == \
            (st["zero_reductions"], st["nonzero_reductions"], st["polynomial_additions"]), (e, strategy)
        assert s["discounted_return"] == st["discounted_return"], (e, strategy)
        assert int(s["gb_hash"]) == polys_hash(gb), (e, strategy)
        if strategy != "random":
            penv.seed(300 + e)
            penv.reset()
            t = penv.run(selection=strategy)
            m = min(len(t), trace.shape[1])   # the reversed strategies run long: the trace is capped, the checksum is not
            assert np.array_equal(trace[e, :m], t[:m, :4]), (e, strategy)
            assert int(s["trace_hash"]) == trace_hash(t), (e, strategy)
    del gen


@pytest.mark.parametrize("strategy", ALL_STRATEGIES)
def test_select_kernel_matches_oracle_row(torch_cuda, strategy):
    """bb_select on live states == the row std::min_element picks (port restatement of buchberger.cpp:160-241)."""
    if strategy == "random":
        pytest.skip("covered by test_all_selection_types_whole_episodes and test_value")
    from deepgroebner_b200.buchberger import BuchbergerEngine
    port = __import__("oracle.oracle", fromlist=["x"]).load_port()
    N = 64
    eng = BuchbergerEngine("3-20-10-uniform", num_envs=N)
    eng.seed(40)
    eng.reset()
    envs = []
    for e in range(N):
        r = port.env("3-20-10-uniform")
        r.seed(40 + e)
        r.reset()
        envs.append(r)
    rng = np.random.default_rng(1)
    for step in range(25):
        rows = eng.select(strategy).cpu().numpy()
        lens = eng.lengths().cpu().numpy()
        acts = np.zeros(N, np.int32)
        for e in range(N):
            if lens[e] == 0:
                continue
            assert rows[e] == envs[e].select(strategy), (step, e)
            acts[e] = rng.integers(lens[e])
            envs[e].step(envs[e].pairs()[acts[e]])
        eng.step(torch_cuda.as_tensor(acts, device="cuda"))


def test_value_matches_reference(torch_cuda):
    """bb_value == BuchbergerEnv::value (buchberger.cpp:332-351) from live mid-episode states, bit-exact doubles;
    the environments themselves are left untouched.  'random' / 'sample' use explicit seeds (the reference reads
    std::random_device there): same buchberger(G, P, ...) overload, seed per rollout."""
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    N = 96
    env = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=128)
    env.seed(np.arange(900, 900 + N))
    refs = []
    for e in range(N):
        r = orc.env("3-20-10-weighted")
        r.seed(900 + e)
        r.reset()
        refs.append(r)
    obs, lengths = env.reset()
    rng = np.random.default_rng(5)
    for step in range(12):
        lens = lengths.cpu().numpy()
        if step in (0, 5, 11):
            before = obs.clone()
            for strat in ("first", "degree", "normal", "sugar", "last", "codegree", "strange", "spice"):
                v = env.value(strat, 0.99).cpu().numpy()
                for e in range(N):
                    assert v[e] == refs[e].value_seeded(strat, 0.99), (step, strat, e)
            v = env.value("random", 0.9, rollouts=5, selection_seed=31).cpu().numpy()
            for e in range(0, N, 4):
                assert v[e] == refs[e].value_seeded("random", 0.9, 31, 5), (step, e)
            if step == 5:
                v = env.value("sample", 0.99, selection_seed=17).cpu().numpy()
                for e in range(0, N, 8):
                    assert v[e] == refs[e].value_seeded("sample", 0.99, 17), (step, e)
            o2, l2 = env.engine.observe(128)
            assert torch_cuda.equal(o2, before) and torch_cuda.equal(l2, lengths)
        acts = np.array([rng.integers(l) if l else 0 for l in lens], dtype=np.int32)
        for e in range(N):
            if lens[e]:
                refs[e].step(refs[e].pairs()[acts[e]])
        (obs, lengths), _, _, _ = env.step(torch_cuda.as_tensor(acts, device="cuda"))


def test_value_single_env_matches_cython_docstring_case(torch_cuda):
    """SURVEY 8(c): seed 123, reset, step(3) (reward -1.0), value('degree', 0.99) == -123.7032989562525."""
    from deepgroebner_b200 import LeadMonomialsEnv
    env = LeadMonomialsEnv("3-20-10-weighted", k=2)
    env.seed(123)
    env.reset()
    _, reward, _, _ = env.step(3)
    assert reward == -1.0
    assert env.value("degree", 0.99) == -123.7032989562525


def test_copy_is_deep_and_includes_the_ideal_stream(torch_cuda):
    """copy() (wrapped.pyx:35-38, buchberger.cpp:279-283): the copy continues identically and independently, and its
    next reset() draws the same next ideal as the original's."""
    from deepgroebner_b200 import LeadMonomialsEnv
    a = LeadMonomialsEnv("3-20-10-weighted", k=2)
    a.seed(5)
    a.reset()
    a.step(1)
    b = a.copy()
    sa, ra, da, _ = a.step(2)
    sb, rb, db, _ = b.step(2)
    assert np.array_equal(sa, sb) and ra == rb and da == db
    sa2, _, _, _ = a.step(0)
    assert np.array_equal(b._state(), sb)          # stepping a did not move b
    assert np.array_equal(a.reset(), b.reset())    # same generator stream position
    assert a.value("normal") == b.value("normal")


def test_cyclic6_seeded_random_episodes(torch_cuda):
    """BASELINE configs[4]: cyclic-6 over GF(32003), 256 episodes under seeded Random selection -- long reductions
    (dividends of hundreds of terms), pair sets beyond 1000 entries, every environment on a different trajectory.
    EVERY record field of EVERY episode equals the unmodified reference env driven with choice() on the same
    minstd_rand0 stream (ref_run_records); the first 8 are also tied to the reference's own buchberger(F, Random, ...,
    seed) loop (reduction counts, additions, discounted return, reduced Groebner basis).  Degree is checked with its
    full pair sequence."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    episodes, sel_seed = 256, 1234
    eng = BuchbergerEngine("cyclic-6", num_envs=episodes)
    stats, _ = eng.run_episodes("random", episodes=episodes, compute_gb=True, selection_seed=sel_seed, gamma=0.99)
    assert (stats["status"] == 2).all()
    assert_records_equal(stats, reference_records("cyclic-6", "random", episodes, sel_seed0=sel_seed), "cyclic-6/random")
    assert len(set(stats["steps"].tolist())) > episodes // 4   # the episodes really are different trajectories
    env = orc.env("cyclic-6")
    F, _ = env.reset()
    for e in range(8):
        gb, st = orc.buchberger(F, selection="random", gamma=0.99, seed=sel_seed + e)
        s = stats[e]
        assert (s["zero_reductions"], s["nonzero_reductions"], s["additions"]) == \
            (st["zero_reductions"], st["nonzero_reductions"], st["polynomial_additions"]), e
        assert s["discounted_return"] == st["discounted_return"], e
        assert (s["gb_polys"], s["gb_terms"]) == (len(gb), sum(len(g) for g in gb))
        assert int(s["gb_hash"]) == polys_hash(gb), e
    stats, trace = eng.run_episodes("degree", episodes=2, compute_gb=True, trace_episodes=2, trace_cap=4096)
    t = env.run(selection="degree")
    for e in range(2):
        assert stats["steps"][e] == len(t) and np.array_equal(trace[e, :len(t)], t[:, :4])
        assert int(stats["trace_hash"][e]) == trace_hash(t) and int(stats["basis_hash"][e]) == polys_hash(env.basis())


def test_sharded_blocks_equal_one_run(torch_cuda):
    """SURVEY 8(e): an episode's record does not depend on how the episode range is cut into per-GPU blocks --
    run_sharded over one rank == the concatenation of the blocks that 2 and 3 ranks would run."""
    from deepgroebner_b200 import sharding
    from deepgroebner_b200.buchberger import BuchbergerEngine
    total = 301
    eng = BuchbergerEngine("3-20-10-uniform", num_envs=128)
    whole = sharding.run_sharded(eng, "normal", total, seed_base=50, compute_gb=True)
    assert whole.shape == (total,) and (whole["status"] == 2).all()
    for ws in (2, 3):
        parts = []
        for r in range(ws):
            first, count = sharding.shard_range(total, r, ws)
            st, _ = eng.run_episodes("normal", episodes=count, seed_base=50 + first, compute_gb=True)
            parts.append(st)
        cat = np.concatenate(parts)
        for f in ("steps", "additions", "trace_hash", "basis_hash", "gb_hash", "discounted_return", "rerolls"):
            assert np.array_equal(cat[f], whole[f]), (ws, f)
    assert sharding.summarize(whole)["finished"] == total


@pytest.mark.parametrize("name,strategy", [("cyclic-5", "normal"), ("cyclic-6", "degree"), ("cyclic-6", "random"),
                                           ("3-20-10-weighted", "degree")])
def test_cta_per_environment_runner_equals_warp_runner(torch_cuda, name, strategy):
    """bb_set_wide: reduce() by streams (bb_streams.cuh: the dividend is never materialised, one round per lead term) and
    the materialising runner (warp_merge / warp_reduce) produce bit-identical episode records -- pair sequence checksum,
    additions, final basis, reduced Groebner basis, discounted return -- and traffic counters.  Modes 1-3 and 7 run the
    streams with one CTA per environment (bb_wide.cuh): 1 = 256 register slots + the shared-memory table, 2 / 3 = 6 / 48
    slots (consolidation of the dividend into a scratch list every few additions), 7 = 8 register slots + the table (the
    shared-memory path on every step), 8 = 32 instead of 256 reducers in the control warp's registers (the scan of the
    rest of the reducer list in memory).  Modes 4-6 run one warp per environment with every stream in registers
    (bb_rstreams.cuh): 128 / 6 / 48 slots.  terms_read / terms_written (|h| per addition) exist only where h is
    materialised."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    episodes = 12
    eng = BuchbergerEngine(name, num_envs=episodes, **({} if name.startswith("cyclic") else dict(max_poly_terms=256)))
    out = {}
    for mode in (0, 1, 2, 3, 4, 5, 6, 7, 8):
        eng.set_wide(mode)
        eng.counters(reset=True)
        stats, trace = eng.run_episodes(strategy, episodes=episodes, seed_base=7, compute_gb=True, selection_seed=99,
                                        trace_episodes=2, trace_cap=4096)
        out[mode] = (stats, trace, eng.counters(reset=True))
    s0, t0, c0 = out[0]
    assert (s0["status"] == 2).all()
    for mode in (1, 2, 3, 4, 5, 6, 7, 8):
        s1, t1, c1 = out[mode]
        for f in s0.dtype.names:
            assert np.array_equal(s0[f], s1[f]), (mode, f)
        assert np.array_equal(t0, t1), mode
        c1 = dict(c1, terms_read=c0["terms_read"], terms_written=c0["terms_written"])
        assert c0 == c1, mode


@pytest.mark.parametrize("dist,kw", [
    ("3-20-10-weighted", {}), ("5-5-10-uniform", {}), ("3-20-10-uniform", dict(elimination="lcm")),
    ("3-20-10-weighted", dict(elimination="none")), ("4-6-8-maximum-homog", dict(sort_input=True)),
    ("3-12-6-weighted-pure", dict(sort_reducers=False)), ("2-9-5-uniform-consts", dict(sort_input=True, sort_reducers=False)),
    ("3-4-16-uniform", {}), ("2-3-3-weighted", {}),
])
def test_episode_preparation_by_thread_equals_by_warp(torch_cuda, dist, kw):
    """bb_set_prepare_mode: the thread-per-episode preparation (generator + reset(), buchberger.cpp:299-315, re-rolls
    included) leaves exactly the state the warp-per-episode one does -- every episode record and every traffic counter
    of the runs that start from it are equal -- and both equal the reference."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    episodes = 600
    eng = BuchbergerEngine(dist, num_envs=256, **kw)
    out = {}
    for by_warp in (False, True):
        eng.set_prepare_mode(by_warp)
        eng.counters(reset=True)
        stats, trace = eng.run_episodes("normal", episodes=episodes, seed_base=11, compute_gb=True, trace_episodes=4,
                                        trace_cap=1024, max_steps=400)
        out[by_warp] = (stats, trace, eng.counters(reset=True))
    (s0, t0, c0), (s1, t1, c1) = out[False], out[True]
    for f in s0.dtype.names:
        assert np.array_equal(s0[f], s1[f]), f
    assert np.array_equal(t0, t1) and c0 == c1
    if not kw.get("sort_input") and kw.get("elimination", "gebauermoeller") == "gebauermoeller":   # lcm / none overflow the binomial pair capacity (flagged, equal in both modes)
        assert_records_equal(s0, reference_records(dist, "normal", episodes, seed0=11, max_steps=400, **kw), dist)
