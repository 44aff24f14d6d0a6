"""GPU parity tests of the round-2 additions: other primes and 7 / 8 variables (tests/test_buchberger.py:328-362,
tests/test_polynomials.cpp:76-86), the C++ nvars quirk of fixed ideals, episode truncation, stream compaction, the
pipelined preparation, global episode offsets of shards, seeding on a stream, value('sample'), the agent on
BuchbergerEnv and the discount kernel.  Everything goes through the C-ABI; the oracle is the checker."""
import numpy as np
import pytest

from test_gpu_parity import assert_records_equal, best_oracle, reference_records, trim

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture()
def port101():
    """The C restatement at p = 101 (the unmodified reference is compiled for 32003 only, polynomials.h:10)."""
    from oracle import oracle as O
    orc = O.load_port()
    orc.set_prime(101)
    yield orc
    orc.set_prime(32003)


def test_prime_101_known_answers(torch_cuda, port101):
    """tests/test_buchberger.py:328-362 (test_LeadMonomialsEnv_0 / _1): F = [y - x^2, z - x^3] over FF(101), grevlex."""
    from deepgroebner_b200 import LeadMonomialsEnv
    from deepgroebner_b200.ideals import FixedIdealGenerator
    F = [[(1, (0, 1, 0)), (100, (2, 0, 0))], [(1, (0, 0, 1)), (100, (3, 0, 0))]]
    env = LeadMonomialsEnv(FixedIdealGenerator(F, 3), prime=101)
    s = env.reset()
    assert np.array_equal(s, [[2, 0, 0, 3, 0, 0]])
    s, _, done, _ = env.step(0)
    assert np.array_equal(s, [[2, 0, 0, 1, 1, 0]]) and not done
    s, _, done, _ = env.step(0)
    assert np.array_equal(s, [[1, 1, 0, 0, 2, 0]]) and not done
    s, _, done, _ = env.step(0)
    assert done
    env = LeadMonomialsEnv(FixedIdealGenerator(F, 3), prime=101, elimination="none")
    s = env.reset()
    assert np.array_equal(s, [[2, 0, 0, 3, 0, 0]])
    s, _, done, _ = env.step(0)
    assert sorted(s.tolist()) == [[2, 0, 0, 1, 1, 0], [3, 0, 0, 1, 1, 0]] and not done
    a = 0 if s[0].tolist() == [3, 0, 0, 1, 1, 0] else 1
    s, _, done, _ = env.step(a)
    assert np.array_equal(s, [[2, 0, 0, 1, 1, 0]]) and not done
    for _ in range(4):
        s, _, done, _ = env.step(0)
    assert done


@pytest.mark.parametrize("strategy", ["degree", "normal"])
def test_prime_101_whole_episodes(torch_cuda, port101, strategy):
    """GF(101) end to end: generator (coefficients uniform on [1, 100]), Barrett reduction and inverse table at another
    modulus, 96 episodes with the full pair sequence against the restatement at the same prime."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from hashing import polys_hash
    E = 96
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=E, prime=101)
    stats, trace = eng.run_episodes(strategy, episodes=E, seed_base=7, compute_gb=True, trace_episodes=E, trace_cap=1024)
    env = port101.env("3-20-10-weighted")
    for e in range(E):
        env.seed(7 + e)
        env.reset()
        t = env.run(selection=strategy)
        assert stats["status"][e] == 2 and stats["steps"][e] == len(t), e
        assert np.array_equal(trace[e, :len(t)], t[:, :4]), e
        assert int(stats["basis_hash"][e]) == polys_hash(env.basis()), e
        assert int(stats["gb_hash"][e]) == polys_hash(env.final_gb()), e


@pytest.mark.parametrize("dist", ["7-2-5-uniform", "8-2-5-uniform", "8-3-4-uniform"])
def test_seven_and_eight_variables(torch_cuda, dist):
    """n = 7 (8-bit fields) and n = 8 (7-bit fields): grevlex on the packed keys (tests/test_polynomials.cpp:76-86 is the
    8-variable order), lcm / divisibility, Gebauer-Moeller and the reduced basis: every record of 2048 episodes equals the
    unmodified reference's."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 2048
    eng = BuchbergerEngine(dist, num_envs=1024)
    for strategy in ("normal", "degree"):
        stats, _ = eng.run_episodes(strategy, episodes=E, seed_base=3, compute_gb=True)
        assert (stats["status"] == 2).all()
        assert_records_equal(stats, reference_records(dist, strategy, E, seed0=3), dist + "/" + strategy)


def test_eight_variable_monomial_order(torch_cuda):
    """tests/test_polynomials.cpp:76-86 on the device: a polynomial's terms come back in descending grevlex order."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from deepgroebner_b200.ideals import FixedIdealGenerator
    orc = best_oracle()
    rng = np.random.default_rng(8)
    monos = {tuple(int(x) for x in rng.integers(0, 4, 8)) for _ in range(40)}
    f = [(int(rng.integers(1, 32003)), m) for m in monos]
    g = [(1, (1, 0, 0, 0, 0, 0, 0, 0)), (1, (0,) * 8)]
    eng = BuchbergerEngine(FixedIdealGenerator([f, g], 8), num_envs=1)
    eng.reset()
    got = eng.basis(0)
    assert got[0] == orc.poly_make(f) and got[1] == orc.poly_make(g)
    keys = [m for _, m in got[0]]
    for a, b in zip(keys, keys[1:]):
        assert orc.mono_cmp(a, b) > 0


def test_cyclic6_observation_and_cxx_nvars_quirk(torch_cuda):
    """SURVEY Q1: the C++ / Cython LeadMonomialsEnv shows 5 variables (20 columns at k = 2) for cyclic-6
    (FixedIdealGenerator::nvars, ideals.cpp:146-154); compat_cxx_nvars=True reproduces its matrices byte for byte, the
    default shows all 6 (24 columns) with the same leading 5 of every monomial."""
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    ref = orc.lm_env("cyclic-6", k=2)
    env = LeadMonomialsEnv("cyclic-6", k=2, compat_cxx_nvars=True)
    full = LeadMonomialsEnv("cyclic-6", k=2)
    s, r, f = env.reset(), ref.reset(), full.reset()
    assert r.shape[1] == 20 and f.shape[1] == 24
    rng = np.random.default_rng(6)
    for step in range(25):
        assert s.shape == r.shape and np.array_equal(s, r), step
        assert f.shape[0] == r.shape[0]
        blocks = f.reshape(f.shape[0], 4, 6)
        assert np.array_equal(blocks[:, :, :5].reshape(f.shape[0], 20), r), step
        a = int(rng.integers(len(r)))
        s, rew, done, _ = env.step(a)
        f, rew_f, done_f, _ = full.step(a)
        r, rew_r, done_r, _ = ref.step(a)
        assert rew == rew_r == rew_f and done == done_r == done_f


def test_max_episode_length_truncates_like_pg(torch_cuda):
    """pg.py:470-471: the episode ends once episode_length > max_episode_length, i.e. after max + 1 steps; the
    environment reports done, goes to `truncated` and (with auto-reset) starts its next episode."""
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    N, L = 64, 6
    env = LeadMonomialsEnv("3-20-10-weighted", k=1, num_envs=N, pmax=64, max_episode_length=L)
    env.seed(np.arange(40, 40 + N))
    env.reset()
    want = []
    ref = orc.env("3-20-10-weighted")
    for e in range(N):
        ref.seed(40 + e)
        ref.reset()
        want.append(len(ref.run(selection="first")))
    first_done = np.full(N, -1)
    for t in range(L + 3):
        _, _, done, _ = env.step(torch.zeros(N, dtype=torch.int32, device="cuda"))   # 'first' selection = row 0
        d = done.cpu().numpy()
        first_done[(first_done < 0) & d] = t + 1
    st = env.engine.stats()
    status = env.engine.status().cpu().numpy()
    for e in range(N):
        assert first_done[e] == min(want[e], L + 1), e
        assert status[e] == (2 if want[e] <= L + 1 else 9), e
        assert st["steps"][e] == min(want[e], L + 1), e
    summ = env.engine.status_summary()
    assert summ["truncated"] == int((status == 9).sum()) and summ["done"] == int((status == 2).sum())
    assert sum(v for k, v in summ.items() if k != "diverged") == N
    # the fused rollout: no episode inside the window is longer than L + 1 steps
    from deepgroebner_b200.rollout import PairsPolicy, collect
    env2 = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=128, pmax=64)
    env2.seed(np.arange(128))
    env2.engine.set_auto_reset(True)
    env2.engine.reset()
    net = PairsPolicy(env2.engine.cols, 32, torch_seed=0, seed=1, device="cuda")
    tb = collect(env2, net, 48, store_obs=False, max_episode_length=L)
    _, lengths = tb.episode_stats()
    assert lengths.numel() > 128 and int(lengths.max()) == L + 1


def test_compaction_is_invisible_and_packs_running_first(torch_cuda):
    """Row N1: bb_compact lists the RUNNING environments first (stable), bb_step takes them in that order; rewards, done
    flags, observations and episode records are those of the uncompacted call."""
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    N = 700
    envs = []
    for on in (True, False):
        env = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=96)
        env.engine.set_compaction(on)
        env.seed(np.arange(N))
        envs.append((env, env.reset()))
    rng = np.random.default_rng(4)
    for step in range(70):
        lens = envs[0][1][1].cpu().numpy()
        acts = torch.as_tensor(np.array([rng.integers(l) if l else 0 for l in lens], dtype=np.int32), device="cuda")
        if step == 0:
            acts[5] = 100000   # a diverged environment (bad action) among the finished ones
        outs = []
        for i, (env, _) in enumerate(envs):
            (obs, lengths), reward, done, _ = env.step(acts)
            outs.append((obs, lengths, reward, done))
            envs[i] = (env, (obs, lengths))
        for a, b in zip(outs[0], outs[1]):
            assert torch.equal(a, b), step
        if step % 23 == 5:
            eng = envs[0][0].engine
            lst = eng.compact().cpu().numpy()
            status = eng.status().cpu().numpy()
            running = np.nonzero(status == 1)[0]
            idle = np.nonzero(status != 1)[0]
            assert lst[0] == len(running)
            assert np.array_equal(lst[1:1 + len(running)], running) and np.array_equal(lst[1 + len(running):], idle)
    a, b = envs[0][0].engine.stats(), envs[1][0].engine.stats()
    for f in ("steps", "additions", "status", "trace_hash", "nbasis"):
        assert np.array_equal(a[f], b[f]), f
    summ = envs[0][0].engine.status_summary()
    assert summ["bad_action"] == 1 and summ["diverged"] == 1 and summ["done"] > 0
    assert summ["done"] + summ["running"] + summ["bad_action"] == N


def test_prepared_batches_pipeline(torch_cuda):
    """bb_prepare on a side stream + bb_run: the records of a prepared call equal those of a plain one; a prepared batch
    that does not match the next run is ignored; back-to-back pipelined calls on alternating staging sets stay exact."""
    torch = torch_cuda
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 3000
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=1024)
    side = torch.cuda.Stream()
    want = {b: reference_records("3-20-10-weighted", "degree", E, seed0=b) for b in (0, 5000, 9000)}
    seeds = torch.arange(5000, 5000 + E, dtype=torch.int32, device="cuda")
    # plain, then prepared with explicit seeds, then a prepared batch that is NOT the one run next
    stats, _ = eng.run_episodes("degree", episodes=E, seed_base=0, compute_gb=True)
    assert_records_equal(stats, want[0], "plain")
    side.wait_stream(torch.cuda.current_stream())   # the seeds were written on this stream
    with torch.cuda.stream(side):
        eng.prepare_episodes(E, seeds=seeds)
    stats, _ = eng.run_episodes("degree", episodes=E, seeds=seeds, compute_gb=True)
    assert_records_equal(stats, want[5000], "prepared")
    with torch.cuda.stream(side):
        eng.prepare_episodes(E, seed_base=123)
    stats, _ = eng.run_episodes("degree", episodes=E, seed_base=9000, compute_gb=True)
    assert_records_equal(stats, want[9000], "mismatched prepare ignored")
    # pipeline: the batch of call i + 1 is prepared while call i runs
    bases = [0, 9000, 0, 9000, 0]
    bufs = []
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eng.prepare_episodes(E, seed_base=bases[0])
    for i, b in enumerate(bases):
        if i + 1 < len(bases):
            with torch.cuda.stream(side):
                eng.prepare_episodes(E, seed_base=bases[i + 1])
        buf, _ = eng.run_episodes("degree", episodes=E, seed_base=b, compute_gb=True, to_host=False)
        bufs.append(buf.clone())
    torch.cuda.synchronize()
    from deepgroebner_b200 import _lib
    for b, buf in zip(bases, bufs):
        assert_records_equal(buf.cpu().numpy().view(np.dtype(_lib.STATS_DTYPE)), want[b], "pipelined %d" % b)
    eng.set_timing(True)
    eng.run_episodes("degree", episodes=E, seed_base=0)
    prep_ms, run_ms = eng.last_run_ms()
    assert 0.0 < prep_ms < 50.0 and 0.0 < run_ms < 500.0


def test_shards_follow_the_global_episode_index(torch_cuda):
    """ADVICE r1: with 'random' selection (per-episode selection seeds) and with several staged fixed ideals, episode g of a
    job has the same record whether it runs in one block or as part of a rank's shard."""
    from deepgroebner_b200 import sharding
    from deepgroebner_b200.buchberger import BuchbergerEngine
    total = 157
    eng = BuchbergerEngine("3-20-10-uniform", num_envs=64)
    whole = sharding.run_sharded(eng, "random", total, seed_base=10, compute_gb=True, selection_seed=77)
    assert_records_equal(whole, reference_records("3-20-10-uniform", "random", total, seed0=10, sel_seed0=77),
                         "random, one block")
    for ws in (2, 3):
        parts = []
        for r in range(ws):
            first, count = sharding.shard_range(total, r, ws)
            eng.set_episode_offset(first)
            st, _ = eng.run_episodes("random", episodes=count, seed_base=10 + first, compute_gb=True, selection_seed=77)
            eng.set_episode_offset(0)
            parts.append(st.copy())
        assert_records_equal(np.concatenate(parts), whole, "random, %d shards" % ws)
    # fixed ideals: three different staged ideals, episode g replays ideal g mod 3
    orc = best_oracle()
    env = orc.env("3-20-10-weighted")
    ideals = []
    for s in (1, 2, 3):
        env.seed(s)
        ideals.append(trim(env.reset()[0], 3))
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=16)
    eng.set_ideals(ideals)
    whole, _ = eng.run_episodes("normal", episodes=10, compute_gb=True)
    assert len(set(whole["basis_hash"][:3].tolist())) == 3 and np.array_equal(whole["basis_hash"][:3], whole["basis_hash"][3:6])
    eng.set_episode_offset(4)
    part, _ = eng.run_episodes("normal", episodes=6, compute_gb=True)
    eng.set_episode_offset(0)
    assert_records_equal(part, whole[4:], "staged ideals, offset 4")


def test_staged_prefix_is_what_run_replays(torch_cuda):
    """ADVICE r1: bb_run replays staged ideal e mod (number of staged ideals), not e mod num_envs; a handle without any
    ideal refuses to run instead of reporting empty episodes."""
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    cyc3 = trim(orc.cyclic(3), 3)
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=8)
    eng.set_ideals([cyc3])   # ONE staged ideal in a handle of 8 environments
    stats, _ = eng.run_episodes("first", episodes=5, compute_gb=True)
    env = orc.env("cyclic-3")
    env.reset()
    t = env.run(selection="first")
    assert (stats["status"] == 2).all() and (stats["steps"] == len(t)).all() and len(set(stats["gb_hash"].tolist())) == 1
    eng2 = BuchbergerEngine("3-20-10-weighted", num_envs=4)
    eng2.set_ideals([cyc3], env_ids=[2])   # environment 0 holds nothing
    with pytest.raises(_lib.BBError):
        eng2.run_episodes("first", episodes=2)


def test_seed_on_stream_and_reseed_every_episode(torch_cuda):
    """seed() is one kernel on the current stream (no allocation, no synchronisation): the reference pattern of seeding
    before every episode (randomized_agent.py:141-142) gives the reference's episodes, explicit per-environment seeds too."""
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    env = LeadMonomialsEnv("3-20-10-weighted", k=2)
    ref = orc.lm_env("3-20-10-weighted", k=2)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for seed in (3, 1, 4, 1, 5):
            env.seed(seed)
            ref.seed(seed)
            assert np.array_equal(env.reset(), ref.reset())
    envN = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=5, pmax=64)
    for rep in range(3):
        seeds = np.array([9, 2, 6, 5, 3]) + rep
        envN.seed(seeds)
        obs, lengths = envN.reset()
        for e in range(5):
            ref.seed(int(seeds[e]))
            r = ref.reset()
            assert np.array_equal(obs[e, :int(lengths[e])].cpu().numpy(), r)


def test_value_sample_runs_the_hundred_random_rollouts(torch_cuda):
    """ADVICE r1: value('sample') = max over 1 Degree + 100 Random rollouts (buchberger.cpp:333-341) by default."""
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    N = 24
    env = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=128)
    env.seed(np.arange(300, 300 + N))
    env.reset()
    v_sample = env.value("sample", 0.99, selection_seed=17).cpu().numpy()
    v_degree = env.value("degree", 0.99).cpu().numpy()
    for e in range(N):
        r = orc.env("3-20-10-weighted")
        r.seed(300 + e)
        r.reset()
        assert v_sample[e] == r.value_seeded("sample", 0.99, 17), e
        assert v_sample[e] == r.value_seeded("sample", 0.99, 17, 101), e
    assert (v_sample >= v_degree).all() and (v_sample > v_degree).any()


def test_agent_drives_both_environment_classes(torch_cuda):
    """ADVICE r1: BuchbergerAgent.act returns what the environment's step() takes: a pair for BuchbergerEnv
    (buchberger.py:397-439), a row for LeadMonomialsEnv."""
    from deepgroebner_b200 import BuchbergerAgent, BuchbergerEnv, LeadMonomialsEnv
    orc = best_oracle()
    for strategy in ("degree", "normal"):
        agent = BuchbergerAgent(strategy)
        ref = orc.env("3-20-10-weighted")
        ref.seed(11)
        ref.reset()
        t = ref.run(selection=strategy)
        env = BuchbergerEnv("3-20-10-weighted")
        env.seed(11)
        env.reset()
        total, steps, done = 0.0, 0, False
        while not done:
            a = agent.act(env)
            assert tuple(a) == (int(t[steps, 0]), int(t[steps, 1]))
            _, r, done, _ = env.step(a)
            total += r
            steps += 1
        assert steps == len(t) and total == -float(t[:, 2].sum())
        lm = LeadMonomialsEnv("3-20-10-weighted", k=1)
        lm.seed(11)
        lm.reset()
        steps, done = 0, False
        while not done:
            _, r, done, _ = lm.step(agent.act(lm))
            assert r == -float(t[steps, 2])
            steps += 1
        assert steps == len(t)
    envN = BuchbergerEnv("3-20-10-weighted", num_envs=6, pmax=256)
    envN.seed(np.arange(6))
    envN.reset()
    agent = BuchbergerAgent("degree")
    for _ in range(5):
        (pairs, lengths), reward, done, _ = envN.step(agent.act(envN))
    assert (reward.cpu().numpy() <= 0.0).all() and (reward.cpu().numpy() <= -1.0).any()


def test_discount_kernel_equals_the_host_restatement(torch_cuda):
    """bb_discount (rewards-to-go and GAE of pg.py:18-78 as one kernel each) == the torch restatement, bit for bit."""
    torch = torch_cuda
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from deepgroebner_b200.rollout import compute_advantages, discount_rewards
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=1)
    g = torch.Generator().manual_seed(0)
    N, T = 257, 61
    rewards = -torch.randint(1, 9, (N, T), generator=g).to(torch.float32)
    values = torch.randn((N, T), generator=g)
    done = torch.rand((N, T), generator=g) < 0.1
    a = discount_rewards(rewards, done, 0.99)
    b = discount_rewards(rewards.cuda(), done.cuda(), 0.99, eng)
    assert torch.equal(a, b.cpu())
    a = compute_advantages(rewards, values, done, 0.99, 0.97)
    b = compute_advantages(rewards.cuda(), values.cuda(), done.cuda(), 0.99, 0.97, eng)
    assert torch.equal(a, b.cpu())


def test_runners_of_two_batches_overlap_on_two_streams(torch_cuda):
    """bb_run on alternating streams: the CTAs of batch i + 1 move in while batch i drains (the call on the second stream
    runs in a second bank of environment slots), the preparation runs two batches ahead on a third stream (ring of three
    staging sets).  Every record of every batch equals the reference's."""
    torch = torch_cuda
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    E = 6000
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=min(resident_envs(0, 3), E))
    bases = [0, 7000, 14000, 0, 7000, 14000, 0]
    want = {b: reference_records("3-20-10-weighted", "degree", E, seed0=b) for b in set(bases)}
    main, alt, side = torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.Stream()
    outs = [torch.empty(E * 72, dtype=torch.uint8, device="cuda") for _ in bases]
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        eng.prepare_episodes(E, seed_base=bases[0])
        eng.prepare_episodes(E, seed_base=bases[1])
    for i, b in enumerate(bases):
        with torch.cuda.stream(main if i % 2 == 0 else alt):
            eng.run_episodes("degree", episodes=E, seed_base=b, compute_gb=True, to_host=False, out=outs[i])
        if i + 2 < len(bases):
            with torch.cuda.stream(side):
                eng.prepare_episodes(E, seed_base=bases[i + 2])
    torch.cuda.synchronize()
    for i, b in enumerate(bases):
        assert_records_equal(outs[i].cpu().numpy().view(np.dtype(_lib.STATS_DTYPE)), want[b], "batch %d (seed base %d)" % (i, b))
    c = eng.counters()
    assert c["episodes"] == E * len(bases)
    # a plain run afterwards works and is exact
    stats, _ = eng.run_episodes("degree", episodes=E, seed_base=7000, compute_gb=True)
    assert_records_equal(stats, want[7000], "plain run after the pipeline")


def test_single_environment_server_equals_launch_per_call(torch_cuda):
    """bb_set_serve: a one-environment handle answers reset() / step() through a resident warp and a mailbox in mapped host
    memory.  Same states, rewards and done flags as one kernel launch per call and as the reference, across re-seeding,
    value() and copy() in between (they join the server), an idle period longer than the warp's patience (it leaves and a
    new instance picks the pending command up), a larger state matrix, auto-reset and truncation."""
    import time
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    served = LeadMonomialsEnv("3-20-10-weighted", k=2, pmax=64)
    plain = LeadMonomialsEnv("3-20-10-weighted", k=2, pmax=64)
    plain.engine.set_serve(False)
    ref = orc.lm_env("3-20-10-weighted", k=2)
    rng = np.random.default_rng(12)
    steps = 0
    for ep, seed in enumerate((5, 6, 7, 5, 8, 9)):
        for env in (served, plain, ref):
            env.seed(seed)
        s, p, r = served.reset(), plain.reset(), ref.reset()
        done = False
        while not done:
            assert np.array_equal(s, r) and np.array_equal(p, r)
            a = int(rng.integers(len(r)))
            if steps % 17 == 5:
                assert served.value("degree") == plain.value("degree") == ref.value("degree")
            if steps % 23 == 7:
                time.sleep(0.03)   # longer than the resident warp waits for a command
            if steps % 29 == 11:
                twin = served.copy()
                t_s, t_r, t_d, _ = twin.step(a)
            s, rs, ds, _ = served.step(a)
            p, rp, dp, _ = plain.step(a)
            r, rr, done, _ = ref.step(a)
            if steps % 29 == 11:
                assert np.array_equal(t_s, s) and t_r == rs and t_d == ds
            assert rs == rp == rr and ds == dp == done
            steps += 1
    assert steps > 200
    cs, cp = served.engine.counters(), plain.engine.counters()
    for k in ("env_steps", "additions", "episodes", "lms_scanned", "obs_rows"):
        assert cs[k] == cp[k], k
    # a state matrix with more rows than the mailbox was sized for; auto-reset and truncation through the server
    wide = LeadMonomialsEnv("3-20-10-weighted", k=2, pmax=16, max_episode_length=4)
    wide.engine.set_auto_reset(True)
    wide.seed(3)
    s = wide.reset()
    wide.pmax = 512
    dones = 0
    for t in range(40):
        s, rew, done, _ = wide.step(0)
        dones += done
        assert len(s) > 0   # auto-reset: the state after a finished episode is the next episode's first state
    assert dones >= 8       # cut after max + 1 = 5 steps (or finished earlier)
    assert wide.engine.status_summary()["running"] == 1


def test_prefetched_resets_draw_the_same_episodes(torch_cuda):
    """bb_set_prefetch: resets served from per-environment queues of prepared episodes (filled by one thread per environment
    from the environment's own stream) give the states, rewards, done flags and records of resets through the generator --
    across auto-reset, explicit masked resets, re-seeding of some environments mid-run, a copy into the batch and queues that
    run empty (depth 1) -- and the reference's first states."""
    torch = torch_cuda
    from deepgroebner_b200 import LeadMonomialsEnv
    orc = best_oracle()
    N = 192
    envs = []
    for depth in (8, 1, 0):
        env = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=96)
        env.engine.set_prefetch(depth)
        env.engine.set_auto_reset(True)
        env.seed(np.arange(70, 70 + N))
        envs.append(env)
    states = [env.reset() for env in envs]
    ref = orc.lm_env("3-20-10-weighted", k=2)
    for e in (0, 17, N - 1):
        ref.seed(70 + e)
        r = ref.reset()
        assert np.array_equal(states[0][0][e, :len(r)].cpu().numpy(), r)
    rng = np.random.default_rng(9)
    donor = LeadMonomialsEnv("3-20-10-weighted", k=2, num_envs=N, pmax=96)
    donor.seed(np.arange(900, 900 + N))
    donor.reset()
    for step in range(150):
        for a, b in zip(states[0], states[1]):
            assert torch.equal(a, b), step
        for a, b in zip(states[0], states[2]):
            assert torch.equal(a, b), step
        lens = states[0][1].cpu().numpy()
        acts = torch.as_tensor(np.array([0 if step % 3 else rng.integers(l) for l in lens], dtype=np.int32), device="cuda")
        outs = []
        for i, env in enumerate(envs):
            if step == 40:      # new streams for a third of the environments: their prepared episodes are dropped
                seeds = np.arange(70, 70 + N)
                seeds[::3] += 5000
                env.seed(seeds)
            if step == 60:      # an explicit reset of some environments
                mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
                mask[5:50] = 1
                env.engine.reset(mask)
            if step == 80:      # a foreign environment copied in: its stream comes with it
                env.engine.copy_env(7, donor.engine, 3)
            if step in (60, 80):
                states[i] = env.engine.observe(96)
            (obs, lengths), reward, done, _ = env.step(acts)
            outs.append((reward, done))
            states[i] = (obs, lengths)
        if step in (60, 80):
            continue   # the action tensor was built for the states before the reset / copy
        for a, b in zip(outs[0], outs[1]):
            assert torch.equal(a, b), step
        for a, b in zip(outs[0], outs[2]):
            assert torch.equal(a, b), step
    sa, sb, sc = (env.engine.stats() for env in envs)
    for f in ("steps", "additions", "status", "trace_hash", "nbasis", "rerolls"):
        assert np.array_equal(sa[f], sb[f]) and np.array_equal(sa[f], sc[f]), f
    ca, cc = envs[0].engine.counters(), envs[2].engine.counters()
    for k in ("env_steps", "additions", "episodes", "lms_scanned"):
        assert ca[k] == cc[k], k
    assert ca["episodes"] > N   # plenty of auto-resets happened
