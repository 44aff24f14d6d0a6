"""CPU checks of the fused rollout's row store (bb_rollout_rows): the exported symbol and its ctypes prototype against
the header, and TrajectoryBatch in rows mode on hand-built tensors -- row offsets, halted environments, the
finished-trajectory and single-row rules, and batches() padding each minibatch to its own largest state."""
import ctypes as C
import os
import re

import pytest
import torch

from deepgroebner_b200.rollout import PairsPolicy, TrajectoryBatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLS, PMAX = 6, 7


def header_params(name):
    """ctypes types of the parameters of `name` as declared in include/bbenv.h."""
    hdr = open(os.path.join(ROOT, "include", "bbenv.h")).read()
    m = re.search(r"\bint %s\(([^)]*)\);" % name, hdr)
    assert m, name
    kinds = {"uint64_t": C.c_uint64, "int64_t": C.c_int64, "double": C.c_double, "int": C.c_int}
    out = []
    for p in m.group(1).split(","):
        p = " ".join(p.split())
        out.append(C.c_void_p if "*" in p else kinds[p.split()[0]])
    return out


def test_rollout_rows_is_exported_with_the_header_prototype():
    from deepgroebner_b200 import _lib
    assert "bb_rollout_rows" in _lib.EXPORTS
    want = header_params("bb_rollout_rows")
    # bb_rollout_value's arguments in the same order, then the row store, then the stream
    assert want[:-3] == header_params("bb_rollout_value")[:-1]
    assert want[-3:] == [C.c_void_p, C.c_int64, C.c_void_p]
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libbbenv.so not built (run __graft_entry__.build())")
    lib = _lib.load()
    assert hasattr(C.CDLL(_lib.LIB_PATH), "bb_rollout_rows")
    assert lib.bb_rollout_rows.argtypes == want and lib.bb_rollout_rows.restype == C.c_int


def hand_built(seed=3, N=5, T=12):
    """The same trajectories in both storage modes: dense obs [N, T, PMAX, COLS] and a row store that holds the
    states of the steps that took an action back to back.  Env 3 stops running at step 8 (auto-reset off: action -1,
    done 1, its |P| still reported); env 4 is halted by the row budget at step 9 (action -1, done 0, lengths 0)."""
    g = torch.Generator().manual_seed(seed)
    lengths = torch.randint(1, PMAX - 1, (N, T), generator=g, dtype=torch.int32)   # dense pmax leaves room
    lengths[0, 2] = lengths[1, 5] = 1          # single-row states: never training samples
    actions = (torch.rand((N, T), generator=g) * lengths).to(torch.int32)
    done = torch.rand((N, T), generator=g) < 0.25
    done[:, T - 1] = True
    done[0, :] = False                           # env 0: one unfinished trajectory -- nothing of it is kept
    actions[3, 8:], done[3, 8:] = -1, True
    actions[4, 9:], done[4, 9:], lengths[4, 9:] = -1, False, 0
    done[4, 5], done[4, 6:9] = True, False
    obs = torch.full((N, T, PMAX, COLS), -1, dtype=torch.int32)
    R = 100
    rows = torch.full((N, R, COLS), -7, dtype=torch.int32)
    for e in range(N):
        used = 0
        for t in range(T):
            L = int(lengths[e, t])
            m = torch.randint(0, 9, (L, COLS), generator=g, dtype=torch.int32)
            obs[e, t, :L] = m
            if actions[e, t] >= 0:
                rows[e, used:used + L] = m
                used += L
    base = dict(actions=actions, logp=-torch.rand((N, T), generator=g), lengths=lengths, done=done.to(torch.uint8),
                reward=-torch.randint(1, 6, (N, T), generator=g).float())
    return dict(base, obs=obs), dict(base, rows=rows)


def test_row_offsets_and_halted():
    dense, rowsd = hand_built()
    tb = TrajectoryBatch(rowsd)
    assert tb.halted == 1 and TrajectoryBatch(dense).halted == 0
    N, T = tb.actions.shape
    for e in range(N):
        at = 0
        for t in range(T):
            assert int(tb.offsets[e, t]) == at, (e, t)
            if tb.actions[e, t] >= 0:
                L = int(tb.lengths[e, t])
                assert torch.equal(tb.rows[e, at:at + L], dense["obs"][e, t, :L])
                at += L
    # env 3's steps after it stopped took no action: their |P| takes no rows
    assert int(tb.offsets[3, -1]) == int(tb.lengths[3, :8].sum())


def test_rows_mode_training_set_equals_the_dense_one():
    dense, rowsd = hand_built()
    a, b = TrajectoryBatch(dense), TrajectoryBatch(rowsd)
    ga, gb = a.get(0.9, 0.8), b.get(0.9, 0.8)
    for x, y in zip(ga[1:], gb[1:]):
        assert torch.equal(x, y)
    width = int(gb[0].shape[1])
    assert width < PMAX and (gb[0][:, -1, -1] != -1).any()   # padded to the largest kept state, not to pmax
    assert torch.equal(ga[0][:, :width], gb[0]) and (ga[0][:, width:] == -1).all()
    assert a.dropped_wide == 0 and b.dropped_wide == 0
    # the finished-trajectory rule: nothing of env 0 (no done), of env 3 after it stopped, or of env 4 after its last
    # done (steps 6..8 precede the halt without a done); the single-row rule: (1, 5) is finished but not a sample
    e, t = b.finished.nonzero(as_tuple=True)
    assert not (e == 0).any() and not ((e == 3) & (t >= 8)).any() and not ((e == 4) & (t > 5)).any()
    assert bool(b.finished[1, 5]) and len(ga[1]) == int((b.lengths[b.finished] != 1).sum())


def test_dense_mode_drops_what_rows_mode_keeps():
    dense, rowsd = hand_built()
    dense["obs"] = dense["obs"][:, :, :3].contiguous()   # pmax 3: wider states cannot be stored densely
    a, b = TrajectoryBatch(dense), TrajectoryBatch(rowsd)
    na, nb = len(a.get()[1]), len(b.get()[1])
    assert a.dropped_wide > 0 and b.dropped_wide == 0 and na + a.dropped_wide == nb


@pytest.mark.parametrize("mode", ["obs", "rows"])
@pytest.mark.parametrize("seed", [None, 5])
def test_batches_pad_each_minibatch_to_its_own_largest_state(mode, seed):
    dense, rowsd = hand_built(seed=11, N=6, T=16)
    tb = TrajectoryBatch(dense if mode == "obs" else rowsd)
    full = TrajectoryBatch(dense).get(0.95, 0.9)
    M = len(full[1])
    got = list(tb.batches(5, 0.95, 0.9, seed=seed))
    assert [len(b[1]) for b in got] == [5] * (M // 5) + ([M % 5] if M % 5 else [])
    # every sample exactly once; normalised advantages as in get() (over the whole set)
    def samples(obs, act, lp, adv, rtg):
        return list(zip(adv.tolist(), rtg.tolist(), act.tolist(), lp.tolist(),
                        [tuple(o[o[:, -1] != -1].flatten().tolist()) for o in obs]))

    seen = []
    for obs, act, lp, adv, rtg in got:
        L = (obs[..., -1] != -1).sum(dim=1)
        assert obs.shape[1] == int(L.max())                     # its own largest state
        assert (obs[torch.arange(obs.shape[1])[None, :] >= L[:, None]] == -1).all()
        seen += samples(obs, act, lp, adv, rtg)
    want = samples(*full)
    assert sorted(seen) == sorted(want)
    if seed is None:
        assert seen == want
    assert len({b[0].shape[1] for b in got}) > 1


def test_batches_feed_the_policy_unchanged():
    dense, rowsd = hand_built(seed=4)
    tb = TrajectoryBatch(rowsd)
    net = PairsPolicy(COLS, 32, torch_seed=2)
    for obs, act, lp, adv, rtg in tb.batches(4):
        logp = net.log_probs(obs)
        assert logp.shape == obs.shape[:2]
        L = (obs[..., -1] != -1).sum(dim=1)
        assert torch.allclose(logp.exp().sum(dim=1), torch.ones(len(act)), atol=1e-5)
        assert (act < L).all()
