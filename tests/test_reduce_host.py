"""CPU-side checks of reduce() on the device (bb_reduce): the symbol at the C-ABI, PolyBatch.from_lists (term order against
the oracle's monomial order, refused input), and the grouping of queries by divisor list and back, on hand-built tensors."""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

from deepgroebner_b200.buchberger import PolyBatch, _group_queries, _remainder_batch, _ungroup


def test_reduce_is_exported():
    from deepgroebner_b200 import _lib
    assert "bb_reduce" in _lib.EXPORTS
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libbbenv.so not built (run __graft_entry__.build())")
    assert len(_lib.load().bb_reduce.argtypes) == 17
    assert hasattr(C.CDLL(_lib.LIB_PATH), "bb_reduce")


@pytest.mark.parametrize("n", [1, 3, 5, 8])
def test_from_lists_term_order(port, n):
    rng = np.random.default_rng(n)
    lists = []
    for _ in range(20):
        G = []
        for _ in range(int(rng.integers(0, 4))):
            monos = {tuple(int(x) for x in rng.integers(0, 4, size=n)) for _ in range(int(rng.integers(1, 12)))}
            G.append([(int(rng.integers(1, 32003)), m + (0,) * (8 - n)) for m in monos])
        lists.append(G)
    b = PolyBatch.from_lists(lists, n, "cpu")
    assert b.exps.shape[1] == n and b.stored.all()
    got = b.to_lists()
    for G, H in zip(lists, got):
        assert len(G) == len(H)
        for f, h in zip(G, H):
            pad = [(c, tuple(e) + (0,) * (8 - n)) for c, e in h]
            assert sorted(pad) == sorted(f)   # the same terms ...
            for (_, a), (_, c) in zip(pad, pad[1:]):   # ... strictly descending in the oracle's grevlex
                assert port.mono_cmp(a, c) > 0
            want = sorted(f, key=functools.cmp_to_key(lambda s, t: port.mono_cmp(t[1], s[1])))
            assert pad == want


def test_from_lists_refuses():
    with pytest.raises(ValueError, match="duplicate"):
        PolyBatch.from_lists([[[(1, (1, 0)), (2, (1, 0))]]], 2, "cpu")
    with pytest.raises(ValueError, match="coefficient"):
        PolyBatch.from_lists([[[(0, (1, 0))]]], 2, "cpu")
    with pytest.raises(ValueError, match="coefficient"):
        PolyBatch.from_lists([[[(101, (1, 0))]]], 2, "cpu", prime=101)
    with pytest.raises(ValueError, match="coefficient"):
        PolyBatch.from_lists([[[(-3, (1, 0))]]], 2, "cpu")
    with pytest.raises(ValueError, match="exponents"):
        PolyBatch.from_lists([[[(1, (0, 0, 1))]]], 2, "cpu")
    with pytest.raises(ValueError, match="zero polynomial"):
        PolyBatch.from_lists([[[(1, (1, 0))], []]], 2, "cpu", divisors=True)
    b = PolyBatch.from_lists([[[]], []], 2, "cpu")   # as dividends the zero polynomial and empty entries are fine
    assert b.ep_offsets.tolist() == [0, 1, 1] and b.poly_offsets.tolist() == [0, 0]


def test_group_and_ungroup_queries():
    # five queries (lengths 2, 0, 1, 3, 1) on lists 2, 0, 2, 1, 0
    po = torch.tensor([0, 2, 2, 3, 6, 7])
    ex = torch.arange(14, dtype=torch.int32).view(7, 2)
    cf = torch.tensor([10, 11, 12, 13, 14, 15, 16], dtype=torch.int32)
    which = torch.tensor([2, 0, 2, 1, 0], dtype=torch.int32)
    order, q_off, q_ex, q_cf, wq = _group_queries(po, ex, cf, which)
    assert order.tolist() == [1, 4, 3, 0, 2]   # stable: queries of one list keep their order
    assert wq.tolist() == [0, 0, 1, 2, 2]
    assert q_off.tolist() == [0, 0, 1, 4, 6, 7]
    assert q_cf.tolist() == [16, 13, 14, 15, 10, 11, 12]
    assert q_ex[:, 0].tolist() == [12, 6, 8, 10, 0, 2, 4]
    steps_p = torch.tensor([40, 41, 42, 43, 44], dtype=torch.int32)
    assert _ungroup(order, steps_p)[0].tolist() == [43, 40, 44, 42, 41]


def test_remainder_batch():
    # three queries in two entries (queries 0, 1 | 2); the sink holds query 2 first, then query 0; query 1 was not stored
    where = torch.tensor([[1, 2], [-1, -1], [0, 0]])
    rlen = torch.tensor([3, 5, 2], dtype=torch.int32)
    sx = torch.arange(10, dtype=torch.int32).view(5, 2)
    sc = torch.tensor([20, 21, 22, 23, 24], dtype=torch.int32)
    b = _remainder_batch(where, rlen, sx.view(-1), sc, torch.tensor([0, 2, 3]), torch.tensor([True, True]), 2)
    assert b.ep_offsets.tolist() == [0, 2, 3] and b.poly_offsets.tolist() == [0, 3, 3, 5]
    assert b.coefs.tolist() == [22, 23, 24, 20, 21]
    assert b.exps[:, 1].tolist() == [5, 7, 9, 1, 3]
    assert b.stored.tolist() == [False, True]   # entry 0 lost a query
