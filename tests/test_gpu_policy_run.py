"""Whole episodes with the fused policy head choosing the pairs (bb_run_policy, run_episodes(PairsPolicy)): the same
episodes as the step API driven by bb_policy_pmlp, replayed on the oracle, the selection-independent reduced bases, and
records that do not depend on how the episodes are scheduled.  Every comparison is exact: the head's numerics against a
torch evaluation are test_gpu_policy_rollout.py's subject."""
import ctypes as C

import numpy as np
import pytest

from hashing import polys_hash, trace_hash
from helpers import best_oracle

pytestmark = pytest.mark.gpu

# the record fields the step API keeps per environment (bb_stats)
STEP_FIELDS = ("steps", "additions", "zero_reductions", "nonzero_reductions", "nbasis", "nterms", "status", "rerolls",
               "trace_hash")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def random_net(cols, hidden, torch_seed=5, seed=11):
    """A PairsPolicy with non-zero biases too, so that no two rows tie by construction."""
    import torch
    from deepgroebner_b200.rollout import PairsPolicy
    net = PairsPolicy(cols, hidden=hidden, torch_seed=torch_seed, seed=seed)
    g = torch.Generator().manual_seed(torch_seed + 1)
    net.b1 = torch.rand(hidden, generator=g) * 0.2 - 0.1
    net.b2 = torch.rand(1, generator=g)
    return net


def step_api_episodes(dist, k, net, N, seed_base, counter0, greedy, cap):
    """Episode e = environment e of a handle of N environments seeded seed_base + e, auto-reset off, stepped with
    policy(net, counter=counter0 + t, greedy) + step() until every one is done.  Returns (bb_stats records, trace
    [N, cap, 4] of (i, j, additions, |P| after), -1 padded)."""
    import torch
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine(dist, k=k, num_envs=N)
    eng.seed(seed_base)
    eng.reset()
    pmax = eng.caps["max_pairs"]
    trace = torch.full((N, cap, 4), -1, dtype=torch.int32, device="cuda")
    ar = torch.arange(N, device="cuda")
    pairs, _ = eng.pairs(pmax)
    for t in range(cap):
        running = eng.status() == 1
        if not bool(running.any()):
            break
        actions, _ = eng.policy(net, counter=counter0 + t, greedy=greedy)
        ij = pairs[ar, actions.long()]
        reward, _ = eng.step(actions)
        pairs, lengths = eng.pairs(pmax)
        rows = ar[running]
        trace[rows, t, 0:2] = ij[running]
        trace[rows, t, 2] = (-reward[running]).to(torch.int32)
        trace[rows, t, 3] = lengths[running]
    assert not bool((eng.status() == 1).any()), "an episode is longer than %d steps" % cap
    return eng.stats(), trace.cpu().numpy()


def assert_same_records(a, b, fields=None, what=""):
    for f in fields or a.dtype.names:
        assert np.array_equal(a[f], b[f]), "%s: field %s differs" % (what, f)


SAME_AS_STEP_API = [("3-20-10-weighted", 2, h, g) for h in (32, 128, 256) for g in (False, True)] + \
                   [("5-5-10-uniform", 4, 64, False), ("5-5-10-uniform", 4, 64, True)]


@pytest.mark.parametrize("dist,k,hidden,greedy", SAME_AS_STEP_API)
def test_same_episodes_as_the_step_api(torch_cuda, dist, k, hidden, greedy):
    """512 episodes on a 64-slot handle: traces and records equal the step API's environment by environment.  k = 2 on
    3-20-10-weighted is the tensor-core head (12 columns), 5-5-10-uniform at k = 4 the FMA head (40 columns).  The first
    64 finished episodes of each run (512 over the cases) are replayed on the oracle from their traced pairs: per-step
    additions, length, zero and nonzero reductions, and the hashes of G and of the reduced basis equal the records."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    N, cap, counter0, seed_base = 512, 1024, 1000, 300
    nv = int(dist.split("-")[0])
    net = random_net(2 * nv * k, hidden)
    eng = BuchbergerEngine(dist, k=k, num_envs=64)
    stats, trace = eng.run_episodes(net, episodes=N, seed_base=seed_base, compute_gb=True, trace_episodes=N, trace_cap=cap,
                                    greedy=greedy, policy_counter=counter0)
    assert (stats["status"] == 2).mean() > 0.9
    ref, ref_trace = step_api_episodes(dist, k, net, N, seed_base, counter0, greedy, cap)
    assert np.array_equal(trace, ref_trace)
    assert_same_records(stats, ref, STEP_FIELDS, "step API")
    for e in range(N):
        assert int(stats["trace_hash"][e]) == trace_hash(trace[e, :stats["steps"][e]])

    orc = best_oracle()
    env = orc.env(dist)
    for e in np.nonzero(stats["status"] == 2)[0][:64]:
        env.seed(int(seed_base + e))
        G, P = env.reset()
        zero = nonzero = adds = 0
        T = int(stats["steps"][e])
        for t in range(T):
            i, j, a, n_after = (int(x) for x in trace[e, t])
            assert (i, j) in P, (e, t)
            reward, done = env.step((i, j))
            assert -reward == a, (e, t)
            adds += a
            nG = len(env.basis())
            nonzero, zero = (nonzero + 1, zero) if nG > len(G) else (nonzero, zero + 1)
            G, P = env.basis(), env.pairs()
            assert len(P) == n_after and done == (t == T - 1), (e, t)
        rec = stats[e]
        assert (rec["additions"], rec["zero_reductions"], rec["nonzero_reductions"]) == (adds, zero, nonzero), e
        assert int(rec["basis_hash"]) == polys_hash(env.basis()), e
        assert int(rec["gb_hash"]) == polys_hash(env.final_gb()), e


def test_zero_weights_greedy_is_first(torch_cuda):
    """All logits equal: the argmax is row 0, BB_SELECT_FIRST.  On 16384 episodes every record equals run_episodes('first')
    and the stored reference records of First, and the exported reduced bases are equal."""
    from oracle import golden
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    torch = torch_cuda
    E = 16384
    eng = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=resident_envs(0, 3))
    net = random_net(eng.cols, 256)
    net.W1, net.b1, net.w2, net.b2 = (torch.zeros_like(t) for t in net.parameters())
    stats, _, out = eng.run_episodes(net, episodes=E, greedy=True, return_gb=True)
    first, _, want = eng.run_episodes("first", episodes=E, return_gb=True)
    assert stats.tobytes() == first.tobytes()
    assert out["gb"] == want["gb"]
    assert golden.mismatches(stats, golden.key("3-20-10-weighted", "first", E)) == []


def test_reduced_bases_do_not_depend_on_the_policy(torch_cuda):
    """A reduced Groebner basis does not depend on the pair order: on 16384 sampled-policy episodes every one that ends done
    has Degree's gb_hash, gb_polys and gb_terms, and groebner_bases(selection=net) returns Degree's bases on staged ideals
    and on cyclic-5."""
    from deepgroebner_b200 import cyclic
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    from deepgroebner_b200.strat import groebner_bases
    E = 16384
    eng = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=resident_envs(0, 3))
    net = random_net(eng.cols, 128)
    stats, _ = eng.run_episodes(net, episodes=E, compute_gb=True)
    deg, _ = eng.run_episodes("degree", episodes=E, compute_gb=True)
    done = stats["status"] == 2
    assert done.sum() > E * 0.99
    for f in ("gb_hash", "gb_polys", "gb_terms"):
        assert np.array_equal(stats[f][done], deg[f][done]), f
    assert not np.array_equal(stats["trace_hash"], deg["trace_hash"])

    gen = best_oracle().generator("3-20-10-weighted")
    gen.seed(777)
    ideals = [gen.next() for _ in range(300)]
    want, _ = groebner_bases(ideals, selection="degree")
    for greedy in (False, True):
        got, st = groebner_bases(ideals, selection=random_net(12, 64), greedy=greedy)
        assert got == want and (st["status"] == 2).all()
    c5 = [[(c, tuple(e) + (0,) * 3) for c, e in f] for f in cyclic(5)]
    want, _ = groebner_bases([c5], selection="degree", capacity="general")
    got, _ = groebner_bases([c5], selection=random_net(10, 32), capacity="general")
    assert got == want


def test_records_do_not_depend_on_scheduling(torch_cuda):
    """The same records on a 64-slot handle and on one of resident_envs() slots, after prepare_episodes, on two streams
    (two banks), and as two shards (set_episode_offset) against one whole call.  Sampling: another policy_counter or net.seed
    changes the traces; greedy: it does not."""
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    torch = torch_cuda
    E = 4096
    net = random_net(12, 128)
    small = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=64)
    big = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=resident_envs(0, 3))
    whole, _ = big.run_episodes(net, episodes=E, compute_gb=True, policy_counter=7)
    s64, _ = small.run_episodes(net, episodes=E, compute_gb=True, policy_counter=7)
    assert whole.tobytes() == s64.tobytes()

    big.prepare_episodes(E, seed_base=0)
    prep, _ = big.run_episodes(net, episodes=E, compute_gb=True, policy_counter=7)
    assert prep.tobytes() == whole.tobytes()

    h = E // 2
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bufs = [torch.empty(h * 72, dtype=torch.uint8, device="cuda") for _ in streams]
    got = []
    for r, (s, buf) in enumerate(zip(streams, bufs)):
        with torch.cuda.stream(s):
            big.set_episode_offset(r * h)
            got.append(big.run_episodes(net, episodes=h, seed_base=r * h, compute_gb=True, policy_counter=7, out=buf,
                                        to_host=False)[0])
    big.set_episode_offset(0)
    torch.cuda.synchronize()
    assert b"".join(g.cpu().numpy().tobytes() for g in got) == whole.tobytes()

    parts = []
    for r in range(2):
        small.set_episode_offset(r * h)
        parts.append(small.run_episodes(net, episodes=h, seed_base=r * h, compute_gb=True, policy_counter=7)[0].copy())
    small.set_episode_offset(0)
    assert np.concatenate(parts).tobytes() == whole.tobytes()

    other_counter, _ = big.run_episodes(net, episodes=E, compute_gb=True, policy_counter=8)
    net2 = random_net(12, 128, seed=12)
    other_seed, _ = big.run_episodes(net2, episodes=E, compute_gb=True, policy_counter=7)
    for o in (other_counter, other_seed):
        assert (o["trace_hash"] != whole["trace_hash"]).mean() > 0.5
    g1, _ = big.run_episodes(net, episodes=E, compute_gb=True, policy_counter=7, greedy=True)
    g2, _ = big.run_episodes(net2, episodes=E, compute_gb=True, policy_counter=8, greedy=True)
    assert g1.tobytes() == g2.tobytes()


def test_max_steps_sinks_and_counters(torch_cuda):
    """max_steps cuts episodes (records keep status running), whose G the basis sink stores; a tiny sink makes
    run_episodes repeat the run with the exact totals and return the same polynomials; the counters add up."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 2048
    eng = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=512)
    net = random_net(eng.cols, 64)
    eng.counters(reset=True)
    stats, _, out = eng.run_episodes(net, episodes=E, max_steps=15, compute_gb=True, return_gb=True, return_basis=True)
    c = eng.counters(reset=True)
    cut = stats["status"] == 1
    assert cut.any() and (stats["status"][~cut] == 2).all() and (stats["steps"] <= 15).all()
    assert np.array_equal(out["basis"].stored.cpu().numpy(), np.ones(E, bool))
    assert np.array_equal(out["gb"].stored.cpu().numpy(), ~cut)
    assert c["env_steps"] == int(stats["steps"].sum()) and c["additions"] == int(stats["additions"].sum())
    assert c["episodes"] == E
    s2, _, small = eng.run_episodes(net, episodes=E, max_steps=15, compute_gb=True, return_gb=True, return_basis=True,
                                    gb_capacity=(8, 8), basis_capacity=(8, 8))
    assert s2.tobytes() == stats.tobytes()
    assert small["gb"] == out["gb"] and small["basis"] == out["basis"]


def _run_policy(eng, W, E=64, hidden=32, gb=None, compute_gb=1, episodes=None):
    """bb_run_policy through ctypes: (rc, records bytes)."""
    import torch
    buf = torch.full((E * 72,), 0xAB, dtype=torch.uint8, device="cuda")
    rc = eng.lib.bb_run_policy(eng.h, hidden, *W, 0, 0, 0, E if episodes is None else episodes, 0, None, 0, 0.99,
                               compute_gb, C.c_void_p(buf.data_ptr()), None, 0, 0,
                               C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(gb) if gb is not None else None,
                               None)
    torch.cuda.synchronize()
    return rc, buf.cpu().numpy().tobytes()


def test_argument_errors_do_not_launch(torch_cuda):
    """A policy for other columns, hidden = 48, a NULL weight, bb_set_obs_nvars mode, a gb sink without compute_gb and
    negative episodes fail with a message, and the records buffer is left untouched."""
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine
    torch = torch_cuda
    E = 64
    eng = BuchbergerEngine("3-20-10-weighted", k=2, num_envs=E)
    with pytest.raises(AssertionError):
        eng.run_episodes(random_net(6, 32), episodes=E)
    ws = [t.to("cuda") for t in random_net(12, 32).parameters()]
    W = [C.c_void_p(t.data_ptr()) for t in ws]
    t = [torch.zeros(4096, dtype=torch.int64, device="cuda") for _ in range(5)]
    sink = _lib.BBPolySink(lens_dev=t[0].data_ptr(), exps_dev=t[1].data_ptr(), coefs_dev=t[2].data_ptr(),
                           where_dev=t[3].data_ptr(), used_dev=t[4].data_ptr(), cap_polys=1000, cap_terms=1000)
    cases = [(dict(hidden=48), b"hidden"),
             (dict(W=[W[0], None, W[2], W[3]]), b"null weight"),
             (dict(gb=sink, compute_gb=0), b"compute_gb"),
             (dict(episodes=-1), b"bad argument")]
    for kw, msg in cases:
        rc, rec = _run_policy(eng, kw.pop("W", W), E, **kw)
        assert rc < 0 and msg in eng.lib.bb_last_error(eng.h), kw
        assert rec == b"\xab" * (E * 72)
    eng.set_obs_nvars(2)
    rc, rec = _run_policy(eng, W, E)
    assert rc < 0 and b"obs_nvars" in eng.lib.bb_last_error(eng.h) and rec == b"\xab" * (E * 72)
    assert all(int(x.abs().sum()) == 0 for x in t)
