"""GPU tests of the fused rollout with values (bb_rollout_value): value[e, t] is BuchbergerEnv::value of the state step t
of environment e starts from, bit-exact against the unmodified reference replaying the recorded actions and against the
step-API loop (bb_value, bb_policy_pmlp, bb_step); everything else the rollout does is bb_rollout's, bit for bit."""
import ctypes as C

import numpy as np
import pytest

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


def make_env(dist, N, seed0, k=2, prefetch=None, **caps):
    from deepgroebner_b200 import LeadMonomialsEnv
    env = LeadMonomialsEnv(dist, k=k, num_envs=N, pmax=128, **caps)
    if prefetch is not None:
        env.engine.set_prefetch(prefetch)
    env.seed(np.arange(seed0, seed0 + N))
    env.engine.reset()
    return env


def net_for(env, hidden=128):
    from deepgroebner_b200.rollout import PairsPolicy
    return PairsPolicy(env.engine.cols, hidden, torch_seed=11, seed=5, device="cuda")


def bits(t):
    return t.contiguous().view(dtype=__import__("torch").int64).cpu().numpy()


def step_loop(torch, eng, net, T, counter0, strategy, gamma=0.99, rollouts=None, seed=0, max_steps=0):
    """The same T steps through the step API: bb_value, then bb_policy_pmlp(counter0 + t), then bb_step."""
    N = eng.num_envs
    out = {n: [] for n in ("value", "actions", "logp", "reward", "done", "lengths")}
    for t in range(T):
        out["value"].append(eng.value(strategy, gamma, rollouts=rollouts, selection_seed=seed, max_steps=max_steps).clone())
        out["lengths"].append(eng.lengths().clone())
        a, lp = eng.policy(net, counter=counter0 + t)
        r, d = eng.step(a)
        out["actions"].append(a.clone()); out["logp"].append(lp.clone())
        out["reward"].append(r.clone()); out["done"].append(d.clone())
    torch.cuda.synchronize()
    return {n: torch.stack(v, dim=1) for n, v in out.items()}


def assert_same_as_loop(torch, fused, loop):
    """Values bit for bit (NaN included) everywhere; actions, log-probabilities, rewards and done flags on the steps of
    running environments (the step API writes action 0 where the fused rollout writes -1); lengths everywhere."""
    assert np.array_equal(bits(fused["value"]), bits(loop["value"]))
    assert torch.equal(fused["lengths"], loop["lengths"])
    run = fused["actions"] >= 0
    assert torch.equal(run, loop["lengths"] > 0)
    assert torch.equal(fused["actions"][run], loop["actions"][run])
    assert torch.equal(fused["logp"][run], loop["logp"][run])
    assert torch.equal(fused["reward"][run], loop["reward"][run].to(torch.float32))
    assert torch.equal(fused["done"][run], loop["done"][run])
    assert (fused["value"][~run] == 0.0).all()


def compare_with_loop(torch, dist, N, T, strategy, gamma=0.99, rollouts=None, seed=0, max_steps=0, auto_reset=True,
                      max_len=0, k=2, **caps):
    a, b = make_env(dist, N, 300, k=k, **caps), make_env(dist, N, 300, k=k, **caps)
    net = net_for(a)
    for env in (a, b):
        env.engine.set_auto_reset(auto_reset)
        env.engine.set_max_episode_length(max_len)
    fused = a.engine.rollout(net, T, counter0=77, value=strategy, value_gamma=gamma, value_rollouts=rollouts,
                             value_seed=seed, value_max_steps=max_steps)
    loop = step_loop(torch, b.engine, net, T, 77, strategy, gamma, rollouts, seed, max_steps)
    assert_same_as_loop(torch, fused, loop)
    return fused


# ---- 1. against the unmodified reference

def replay_values(torch, dist, N, T, strategy, gamma=0.99, seed=0, rollouts=None, seed0=10):
    orc = best_oracle()
    env = make_env(dist, N, seed0)
    net = net_for(env)
    env.engine.set_auto_reset(True)
    out = env.engine.rollout(net, T, counter0=1000, value=strategy, value_gamma=gamma, value_rollouts=rollouts,
                             value_seed=seed)
    A, V, L = out["actions"].cpu().numpy(), out["value"].cpu().numpy(), out["lengths"].cpu().numpy()
    R, D = out["reward"].cpu().numpy(), out["done"].cpu().numpy()
    episodes = 0
    for e in range(N):
        r = orc.env(dist)
        r.seed(seed0 + e)
        r.reset()
        for t in range(T):
            P = r.pairs()
            assert L[e, t] == len(P) and 0 <= A[e, t] < len(P)
            assert V[e, t] == r.value_seeded(strategy, gamma, seed, rollouts), (e, t)
            rew, done = r.step(P[A[e, t]])
            assert R[e, t] == rew and bool(D[e, t]) == done
            if done:
                r.reset()
                episodes += 1
    return episodes


def test_degree_values_equal_the_reference(torch_cuda):
    assert replay_values(torch_cuda, "3-20-10-weighted", 48, 160, "degree") > 48
    replay_values(torch_cuda, "5-5-10-uniform", 16, 60, "degree", seed0=40)   # longer episodes: mostly mid-episode states


@pytest.mark.parametrize("strategy,gamma,seed,rollouts", [("first", 0.99, 0, None), ("normal", 0.9, 0, None),
                                                          ("sugar", 0.99, 0, None), ("random", 0.95, 31, 3),
                                                          ("sample", 0.99, 17, None)])
def test_other_strategies_equal_the_reference(torch_cuda, strategy, gamma, seed, rollouts):
    N, T = (8, 4) if strategy == "sample" else (16, 12)
    replay_values(torch_cuda, "3-20-10-weighted", N, T, strategy, gamma, seed, rollouts, seed0=500)


# ---- 2. against the step-API loop

def test_more_than_one_wave_equals_the_step_loop(torch_cuda):
    compare_with_loop(torch_cuda, "3-20-10-weighted", 4096, 24, "degree")


# ---- 3. nothing else changes

@pytest.mark.parametrize("prefetch", [8, 0])
def test_values_change_nothing_else(torch_cuda, prefetch):
    torch = torch_cuda
    N, T = 256, 40
    a, b = make_env("3-20-10-weighted", N, 70, prefetch=prefetch), make_env("3-20-10-weighted", N, 70, prefetch=prefetch)
    net = net_for(a)
    for env in (a, b):
        env.engine.set_auto_reset(True)
        env.engine.counters(reset=True)
    plain = a.engine.rollout(net, T, counter0=5, store_obs=True, pmax=128)
    withv = b.engine.rollout(net, T, counter0=5, store_obs=True, pmax=128, value="degree")
    torch.cuda.synchronize()
    assert set(withv) == set(plain) | {"value"}
    for n in plain:
        assert torch.equal(plain[n], withv[n]), n
    assert (withv["value"] < 0).any()
    oa, ob = a.engine.observe(128), b.engine.observe(128)
    assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1], ob[1])
    assert a.engine.stats().tobytes() == b.engine.stats().tobytes()
    assert a.engine.counters() == b.engine.counters()
    # the next rollout draws the same ideals (random streams and prefetch queues untouched)
    p2 = a.engine.rollout(net, T, counter0=5 + T)
    w2 = b.engine.rollout(net, T, counter0=5 + T)
    for n in p2:
        assert torch.equal(p2[n], w2[n]), n
    assert a.engine.stats().tobytes() == b.engine.stats().tobytes()


# ---- 4. edge cases

def test_auto_reset_off(torch_cuda):
    fused = compare_with_loop(torch_cuda, "3-20-10-weighted", 128, 60, "degree", auto_reset=False)
    idle = fused["actions"] == -1
    assert idle.any() and (fused["value"][idle] == 0.0).all()


def test_truncation_max_steps_and_gamma(torch_cuda):
    fused = compare_with_loop(torch_cuda, "3-20-10-weighted", 128, 40, "degree", max_len=6)
    assert fused["done"].sum() > 128
    compare_with_loop(torch_cuda, "3-20-10-weighted", 128, 24, "degree", max_steps=3)
    compare_with_loop(torch_cuda, "3-20-10-weighted", 128, 24, "normal", gamma=0.5)
    compare_with_loop(torch_cuda, "5-5-10-uniform", 64, 12, "random", gamma=0.9, rollouts=4, seed=3)


def test_overflowing_value_rollouts_are_nan_where_bb_value_puts_them(torch_cuda):
    fused = compare_with_loop(torch_cuda, "3-20-10-weighted", 256, 30, "degree", max_basis=22)
    assert torch_cuda.isnan(fused["value"]).any()


def test_staged_fixed_ideal_on_the_general_preset(torch_cuda):
    compare_with_loop(torch_cuda, "cyclic-5", 8, 10, "degree")


# ---- 5. argument errors

def raw_call(torch, eng, net, T, strategy, value, hidden=None, rollouts=1):
    W1, b1, w2, b2 = net.device_weights(eng.device, eng.cols)
    N = eng.num_envs
    out = dict(actions=torch.full((N, T), 7, dtype=torch.int32, device="cuda"),
               logp=torch.full((N, T), 7.0, device="cuda"), reward=torch.full((N, T), 7.0, device="cuda"),
               done=torch.full((N, T), 7, dtype=torch.uint8, device="cuda"),
               lengths=torch.full((N, T), 7, dtype=torch.int32, device="cuda"))
    v = torch.full((N, max(T, 1)), 7.0, dtype=torch.float64, device="cuda") if value else None
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    rc = eng.lib.bb_rollout_value(eng.h, hidden or net.hidden, p(W1), p(b1), p(w2), p(b2), net.seed, 9, 0, T,
                                  p(out["actions"]), p(out["logp"]), p(out["reward"]), p(out["done"]), p(out["lengths"]),
                                  None, 0, strategy, 0.99, rollouts, 0, 0, p(v), None)
    torch.cuda.synchronize()
    if v is not None:
        out["value"] = v
    return rc, out


def test_argument_errors_write_nothing(torch_cuda):
    torch = torch_cuda
    env = make_env("3-20-10-weighted", 64, 1)
    eng, net = env.engine, net_for(env)
    before = eng.stats().tobytes()
    cases = [(9, True, 128, 4, b"bad value strategy"), (-1, True, 128, 4, b"bad value strategy"),
             (9, False, 128, 4, b"bad value strategy"), (0, True, 128, 0, b"bad argument"),
             (0, True, 96, 4, b"hidden")]
    for strategy, value, hidden, T, msg in cases:
        rc, out = raw_call(torch, eng, net, T, strategy, value, hidden)
        assert rc < 0 and msg in eng.lib.bb_last_error(eng.h), (strategy, value, hidden, T)
        for n, t in out.items():
            assert (t == 7).all(), n
    assert eng.stats().tobytes() == before


def test_null_value_output_is_bb_rollout(torch_cuda):
    torch = torch_cuda
    a, b = make_env("3-20-10-weighted", 64, 1), make_env("3-20-10-weighted", 64, 1)
    net = net_for(a)
    for env in (a, b):
        env.engine.set_auto_reset(True)
    rc, out = raw_call(torch, a.engine, net, 20, 0, False)
    assert rc == 0
    ref = b.engine.rollout(net, 20, counter0=9)
    for n in out:
        assert torch.equal(out[n], ref[n]), n
    assert a.engine.stats().tobytes() == b.engine.stats().tobytes()


# ---- 6. the trainer's path

def test_collect_with_degree_values(torch_cuda):
    torch = torch_cuda
    from deepgroebner_b200.rollout import collect, compute_advantages
    env = make_env("3-20-10-weighted", 64, 900)
    net = net_for(env)
    tb = collect(env, net, 50, value="degree", gamma=0.99)
    assert tb.value is not None and tb.value.dtype == torch.float64 and tb.value.shape == (64, 50)
    adv = compute_advantages(tb.reward, tb.value, tb.done, 0.99, 0.97)
    obs, actions, logp, a, rtg = tb.get(0.99, 0.97, normalize_advantages=False)
    keep = tb.finished
    multi = tb.lengths[keep] != 1
    multi = multi & (tb.lengths[keep] <= tb.obs.shape[2])
    assert torch.equal(a, adv[keep].to(torch.float32)[multi])
    assert not torch.equal(tb.finish(0.99, 0.97)[1], tb.finish(0.99, 0.97, values=torch.zeros_like(tb.value))[1])
