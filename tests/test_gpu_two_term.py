"""The two-term episode runner (k_run<NV, EXPORT, true>, bb_set_two_term): bb_run takes it for binomial distributions, whose
polynomials never have more than two terms, and it must give exactly what the general runner gives -- records, counters and
exported polynomials.  Every other ideal keeps the general runner."""
import numpy as np
import pytest

from hashing import polys_hash, trace_hash
from helpers import best_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def runner_kernels(torch, fn):
    """Names of the k_run instantiations that fn() launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if "k_run<" in e.name})


@pytest.mark.parametrize("dist,strategy,E,seed0", [
    ("3-20-10-weighted", "degree", 4096, 0), ("3-20-10-weighted", "normal", 2048, 11), ("5-5-10-uniform", "sugar", 1024, 3),
    ("3-12-6-weighted-pure", "random", 1024, 5),
])
def test_two_term_runner_equals_general_runner(torch_cuda, dist, strategy, E, seed0):
    """A binomial run through the two-term runner and the same run forced through the general one: identical records,
    identical counters, identical exported reduced bases and final bases; and the profiler sees the runner it expects."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine(dist, num_envs=min(E, 2048))
    runs = {}
    for two in (True, False):
        eng.set_two_term(two)
        eng.counters(reset=True)
        stats, _, out = eng.run_episodes(strategy, episodes=E, seed_base=seed0, selection_seed=77, gamma=0.99,
                                         compute_gb=True, return_gb=True, return_basis=True)
        runs[two] = (stats, eng.counters(reset=True), out)
    (s1, c1, o1), (s0, c0, o0) = runs[True], runs[False]
    assert (s1["status"] == 2).all()
    assert s1.tobytes() == s0.tobytes()
    assert c1 == c0
    assert c1["env_steps"] == int(s1["steps"].sum()) and c1["episodes"] == E
    assert o1["gb"] == o0["gb"] and o1["basis"] == o0["basis"]
    nv = int(dist.split("-")[0])
    for two, flag in ((True, "true"), (False, "false")):
        eng.set_two_term(two)
        names = runner_kernels(torch_cuda, lambda: eng.run_episodes(strategy, episodes=64, seed_base=seed0))
        assert len(names) == 1 and "k_run<%d, false, %s>" % (nv, flag) in names[0], names
    eng.set_two_term(True)


def test_random_polynomial_distribution_keeps_the_general_runner(torch_cuda):
    """Poisson-length random polynomials (RandomIdealGenerator) may have more than two terms: bb_run's warp runner is the
    general k_run, and every episode equals the oracle's."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    dist, strategy, E = "3-6-5-0.5-uniform", "degree", 128
    eng = BuchbergerEngine(dist, num_envs=E)
    eng.set_wide(0)   # these capacities default to the stream runner (k_run_wide); the warp runner is the one with two forms
    names = runner_kernels(torch_cuda, lambda: eng.run_episodes(strategy, episodes=E, seed_base=1000))
    assert len(names) == 1 and "k_run<3, false, false>" in names[0], names
    stats, _ = eng.run_episodes(strategy, episodes=E, seed_base=1000, compute_gb=True)
    orc = best_oracle()
    env = orc.env(dist)
    assert (stats["status"] == 2).all(), np.unique(stats["status"], return_counts=True)
    long_polys = 0
    for e in range(E):
        env.seed(1000 + e)
        env.reset()
        t = env.run(selection=strategy)
        s = stats[e]
        assert s["steps"] == len(t) and s["additions"] == int(t[:, 2].sum()), e
        assert int(s["trace_hash"]) == trace_hash(t), e
        assert int(s["basis_hash"]) == polys_hash(env.basis()), e
        assert int(s["gb_hash"]) == polys_hash(env.final_gb()), e
        long_polys += max(len(g) for g in env.basis()) > 2
    assert long_polys > 0   # the run does exercise polynomials the two-term runner could not hold
