"""GPU tests of the fused rollout's row store (bb_rollout_rows): every state an action is taken from is stored at its own
row count, back to back per environment.  Trajectories are bb_rollout's bit for bit, states equal the dense obs and the
reference replaying the recorded actions (the states a pmax drops included), the budget rule halts an environment and
the next call continues it, and the training set equals the dense one without its drops."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TRAJ = ("actions", "logp", "reward", "done", "lengths")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def best_oracle():
    from oracle import oracle as O
    return O.load_ref() if O.have_ref() else O.load_port()


def make_env(dist, N, seed0, prefetch=None, auto_reset=True):
    from deepgroebner_b200 import LeadMonomialsEnv
    env = LeadMonomialsEnv(dist, k=2, num_envs=N, pmax=128)
    if prefetch is not None:
        env.engine.set_prefetch(prefetch)
    env.seed(np.arange(seed0, seed0 + N))
    env.engine.reset()
    env.engine.set_auto_reset(auto_reset)
    env.engine.counters(reset=True)
    return env


def net_for(env, hidden=128):
    from deepgroebner_b200.rollout import PairsPolicy
    return PairsPolicy(env.engine.cols, hidden, torch_seed=11, seed=5, device="cuda")


def all_states(torch, tb):
    """(e, t) of every step that took an action, and the row store's states there, padded to the widest."""
    e, t = (tb.actions >= 0).nonzero(as_tuple=True)
    return e, t, tb.states(e, t)


def replay(orc, dist, seed0, calls, envs):
    """Replays the recorded actions of consecutive calls through oracle environments: every stored state's rows, every
    reward and done flag.  A step with action -1 and done 0 is a halt: the environment continues in the next call.
    Returns the set of |P| seen."""
    widths = set()
    for e in envs:
        r = orc.lm_env(dist, k=2)
        r.seed(seed0 + e)
        s = r.reset()
        for tb in calls:
            A, R, D = tb.actions[e].cpu().numpy(), tb.reward[e].cpu().numpy(), tb.done[e].cpu().numpy()
            L, off, rows = tb.lengths[e].cpu().numpy(), tb.offsets[e].cpu().numpy(), tb.rows[e].cpu().numpy()
            for t in range(len(A)):
                if A[t] < 0:
                    assert not D[t] and (A[t:] == -1).all() and (L[t:] == 0).all()
                    break
                assert L[t] == len(s) and np.array_equal(rows[off[t]:off[t] + L[t]], s), (e, t)
                widths.add(len(s))
                s, rew, done, _ = r.step(int(A[t]))
                assert R[t] == rew and bool(D[t]) == done, (e, t)
                if done:
                    s = r.reset()
    return widths


# ---- 1. identity with the dense path

@pytest.mark.parametrize("prefetch,auto_reset", [(8, True), (0, True), (8, False)])
def test_rows_change_nothing_else(torch_cuda, prefetch, auto_reset):
    torch = torch_cuda
    from deepgroebner_b200.rollout import TrajectoryBatch
    N, T = 256, 128
    a, b, c = (make_env("3-20-10-weighted", N, 70, prefetch, auto_reset) for _ in range(3))
    net = net_for(a)
    dense = a.engine.rollout(net, T, counter0=5, store_obs=True, pmax=128)
    rows = b.engine.rollout(net, T, counter0=5, rows_per_env=128 * T)
    c.engine.rollout(net, T, counter0=5)
    torch.cuda.synchronize()
    assert int(dense["lengths"].max()) <= 128 and set(rows) == set(TRAJ) | {"rows"}
    for n in TRAJ:
        assert torch.equal(dense[n], rows[n]), n
    tb = TrajectoryBatch(rows)
    assert tb.halted == 0
    if not auto_reset:
        assert (rows["actions"] < 0).any()   # slots whose episode ended stay idle and store nothing
    e, t, st = all_states(torch, tb)
    assert torch.equal(st, dense["obs"][e, t, :st.shape[1]])
    ca, cb, cc = a.engine.counters(), b.engine.counters(), c.engine.counters()   # before observe() counts its rows
    taken = rows["lengths"].to(torch.int64)[rows["actions"] >= 0]
    assert cb.pop("obs_rows") == cc.pop("obs_rows") + int(taken.sum())   # c stores no state
    ca.pop("obs_rows")
    assert ca == cb == cc
    oa, ob = a.engine.observe(128), b.engine.observe(128)
    assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1], ob[1])
    assert a.engine.stats().tobytes() == b.engine.stats().tobytes()


def test_rows_with_values_equal_bb_rollout_value(torch_cuda):
    torch = torch_cuda
    N, T = 256, 128
    a, b = make_env("3-20-10-weighted", N, 90), make_env("3-20-10-weighted", N, 90)
    net = net_for(a)
    ref = a.engine.rollout(net, T, counter0=3, value="degree")
    got = b.engine.rollout(net, T, counter0=3, value="degree", rows_per_env=128 * T)
    torch.cuda.synchronize()
    for n in TRAJ:
        assert torch.equal(ref[n], got[n]), n
    assert torch.equal(ref["value"].view(torch.int64), got["value"].view(torch.int64))
    assert a.engine.stats().tobytes() == b.engine.stats().tobytes()


# ---- 2. states wider than pmax

@pytest.mark.parametrize("dist,pmax,N,T", [("5-5-10-uniform", 32, 32, 128), ("3-20-10-weighted", 16, 48, 96)])
def test_states_wider_than_pmax_are_kept_and_replay_on_the_oracle(torch_cuda, dist, pmax, N, T):
    torch = torch_cuda
    from deepgroebner_b200.rollout import TrajectoryBatch, collect
    env = make_env(dist, N, 400)
    net = net_for(env)
    tb = collect(env, net, T, counter0=7, store_obs=True, pmax=pmax, rows_per_env=True)
    assert tb.rows.shape == (N, max(env.engine.caps["max_pairs"], env.engine.ROWS_PER_STEP * T), env.engine.cols)
    out = dict(actions=tb.actions, logp=tb.logp, reward=tb.reward, done=tb.done, lengths=tb.lengths, obs=tb.obs)
    dense = TrajectoryBatch(out)
    nd, nr = len(dense.get()[1]), len(tb.get()[1])
    assert dense.dropped_wide > 0 and tb.dropped_wide == 0 and nr == nd + dense.dropped_wide
    widths = replay(best_oracle(), dist, 400, [tb], range(N))
    assert max(widths) > pmax


# ---- 3. the budget rule

def test_budget_halts_and_the_next_call_continues(torch_cuda):
    torch = torch_cuda
    from deepgroebner_b200.rollout import TrajectoryBatch
    N, T = 256, 128
    a, b = make_env("3-20-10-weighted", N, 600), make_env("3-20-10-weighted", N, 600)
    net = net_for(a)
    budget = a.engine.caps["max_pairs"]
    free = a.engine.rollout(net, T, counter0=40, store_obs=True, pmax=128, value="degree", rows_per_env=128 * T)
    tight = b.engine.rollout(net, T, counter0=40, value="degree", rows_per_env=budget)
    torch.cuda.synchronize()
    tf, tt = TrajectoryBatch(free), TrajectoryBatch(tight)
    assert tf.halted == 0 and 0 < tt.halted
    halt = (tight["actions"] < 0) & ~tight["done"].bool()
    halted = halt.any(dim=1)
    assert int(halted.sum()) == tt.halted
    th = torch.where(halted, halt.to(torch.int8).argmax(dim=1), torch.full_like(halted, T, dtype=torch.int64))
    before = torch.arange(T, device="cuda")[None, :] < th[:, None]
    for n in TRAJ + ("value",):
        assert torch.equal(tight[n][before], free[n][before]), n
        zero = tight[n][~before]
        assert (zero == (-1 if n == "actions" else 0)).all(), n
    assert torch.equal(tight["value"][~before].view(torch.int64), torch.zeros_like(tight["value"][~before]).view(torch.int64))
    # the halting step's rows did not fit; every earlier state is stored as the free run stores it
    used = (tight["lengths"].to(torch.int64) * (tight["actions"] >= 0)).sum(dim=1)
    hs = halted.nonzero().flatten()
    assert ((used[hs] + free["lengths"][hs, th[hs]]) > budget).all() and (used <= budget).all()
    e, t, st = all_states(torch, tt)
    assert torch.equal(st, tf.states(e, t))
    # the environment keeps the state of the halting step
    o, ln = b.engine.observe(128)
    assert torch.equal(ln[hs], free["lengths"][hs, th[hs]])
    assert torch.equal(o[hs], free["obs"][hs, th[hs]])
    # halted steps are not env-steps
    assert b.engine.counters()["env_steps"] == int((tight["actions"] >= 0).sum()) < a.engine.counters()["env_steps"]
    # a second call continues every environment; the reference replays both calls
    tight2 = TrajectoryBatch(b.engine.rollout(net, T, counter0=40 + T, rows_per_env=budget))
    replay(best_oracle(), "3-20-10-weighted", 600, [tt, tight2], hs[:24].tolist())


# ---- 4. the training set

def test_training_set_equals_the_dense_one(torch_cuda):
    torch = torch_cuda
    from deepgroebner_b200.rollout import TrajectoryBatch, collect
    N, T = 256, 64
    env = make_env("3-20-10-weighted", N, 800)
    net = net_for(env)
    tb = collect(env, net, T, counter0=2, store_obs=True, pmax=128, rows_per_env=128 * T, value="degree")
    dense = TrajectoryBatch({n: getattr(tb, n) for n in ("actions", "logp", "reward", "done", "lengths", "obs", "value")})
    assert tb.halted == 0 and int(tb.lengths.max()) <= 128
    ga, gb = dense.get(0.99, 0.97), tb.get(0.99, 0.97)
    assert dense.dropped_wide == 0 and len(gb[1]) > 1000
    for x, y in zip(ga[1:], gb[1:]):
        assert torch.equal(x, y)
    width = gb[0].shape[1]
    assert width < 128 and torch.equal(ga[0][:, :width], gb[0]) and (ga[0][:, width:] == -1).all()
    for seed in (None, 9):
        keys = []
        for obs, act, lp, adv, rtg in tb.batches(512, 0.99, 0.97, seed=seed):
            L = (obs[..., -1] != -1).sum(dim=1)
            assert obs.shape[1] == int(L.max())
            ref = net.log_probs(obs).gather(1, act.long()[:, None]).squeeze(1)
            assert torch.allclose(ref, lp, rtol=1e-5, atol=1e-5)
            keys.append(torch.stack([adv.double(), rtg.double(), act.double(), lp.double()], dim=1))
        keys = torch.cat(keys)
        want = torch.stack([gb[3].double(), gb[4].double(), gb[1].double(), gb[2].double()], dim=1)
        assert keys.shape == want.shape
        if seed is None:
            assert torch.equal(keys, want)
        else:
            srt = lambda k: k[np.lexsort(k.cpu().numpy().T[::-1])]
            assert torch.equal(srt(keys), srt(want))


# ---- 5. refusals

def raw_call(torch, eng, net, T, rows_per_env, strategy=0, hidden=None, value=True):
    W1, b1, w2, b2 = net.device_weights(eng.device, eng.cols)
    N = eng.num_envs
    out = dict(actions=torch.full((N, T), 7, dtype=torch.int32, device="cuda"),
               logp=torch.full((N, T), 7.0, device="cuda"), reward=torch.full((N, T), 7.0, device="cuda"),
               done=torch.full((N, T), 7, dtype=torch.uint8, device="cuda"),
               lengths=torch.full((N, T), 7, dtype=torch.int32, device="cuda"),
               rows=torch.full((N, max(rows_per_env, 1), eng.cols), 7, dtype=torch.int32, device="cuda"))
    if value:
        out["value"] = torch.full((N, max(T, 1)), 7.0, dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    rc = eng.lib.bb_rollout_rows(eng.h, hidden or net.hidden, p(W1), p(b1), p(w2), p(b2), net.seed, 9, 0, T,
                                 p(out["actions"]), p(out["logp"]), p(out["reward"]), p(out["done"]), p(out["lengths"]),
                                 None, 0, strategy, 0.99, 1, 0, 0, p(out.get("value")), p(out["rows"]), rows_per_env, None)
    torch.cuda.synchronize()
    return rc, out


def test_refusals_enqueue_nothing(torch_cuda):
    torch = torch_cuda
    env = make_env("3-20-10-weighted", 64, 1)
    eng, net = env.engine, net_for(env)
    mp = eng.caps["max_pairs"]
    before, cbefore = eng.stats().tobytes(), eng.counters()
    cases = [dict(rows_per_env=mp - 1, msg=b"max_pairs"), dict(rows_per_env=0, msg=b"max_pairs"),
             dict(rows_per_env=mp - 1, value=False, msg=b"max_pairs"),
             dict(rows_per_env=mp, strategy=9, msg=b"bad value strategy"),
             dict(rows_per_env=mp, strategy=-1, msg=b"bad value strategy"),
             dict(rows_per_env=mp, strategy=9, value=False, msg=b"bad value strategy"),
             dict(rows_per_env=mp, T=0, msg=b"bad argument"), dict(rows_per_env=mp, hidden=96, msg=b"hidden")]
    for c in cases:
        rc, out = raw_call(torch, eng, net, c.get("T", 4), c["rows_per_env"], c.get("strategy", 0), c.get("hidden"),
                           c.get("value", True))
        assert rc < 0 and c["msg"] in eng.lib.bb_last_error(eng.h), c
        for n, t in out.items():
            assert (t == 7).all(), (c, n)
    assert eng.stats().tobytes() == before and eng.counters() == cbefore
    # at the minimum every environment stores the state it starts from
    rc, out = raw_call(torch, eng, net, 4, mp)
    assert rc == 0 and (out["actions"][:, 0] >= 0).all()
