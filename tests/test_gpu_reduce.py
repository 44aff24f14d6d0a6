"""reduce(g, F) on the device (bb_reduce, BuchbergerEngine.reduce, strat.reduce_polynomials): remainders and steps against the
oracle's reduce (and sympy's), bit for bit, on random lists in both scan orders, on every episode's reduced basis of a whole
run, on long polynomials and at another prime; counters, statuses, sinks, argument errors and non-interference."""
import ctypes as C
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 32003


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def orc():
    from helpers import best_oracle
    return best_oracle()


def pad8(f):
    return [(int(c), tuple(int(x) for x in e) + (0,) * (8 - len(e))) for c, e in f]


def engine(n, prime=P, envs=1024, capacity="poly", **caps):
    from deepgroebner_b200.buchberger import BuchbergerEngine
    from deepgroebner_b200.ideals import FixedIdealGenerator
    return BuchbergerEngine(FixedIdealGenerator([[(1, (0,) * n)]], n), num_envs=envs, prime=prime, capacity=capacity, **caps)


def rand_poly(rng, n, nterms, maxexp, prime=P):
    monos = set()
    while len(monos) < nterms:
        monos.add(tuple(int(x) for x in rng.integers(0, maxexp + 1, size=n)))
    return [(int(rng.integers(1, prime)), m) for m in monos]


def canon(orc, f):
    return orc.poly_make(pad8(f))


def by_lead(orc, F):
    """F stable-sorted by ascending lead monomial (the order of G_ under sort_reducers)."""
    return sorted(F, key=functools.cmp_to_key(lambda a, b: orc.mono_cmp(a[0][1], b[0][1])))


def batch(lists, n, prime=P, divisors=False):
    from deepgroebner_b200.buchberger import PolyBatch
    return PolyBatch.from_lists(lists, n, "cuda:0", prime=prime, divisors=divisors)


def test_known_answers(torch_cuda, orc):
    """test_buchberger.cpp:58-77, the pairs of test_oracle_known_answers.py::test_reduce."""
    from deepgroebner_b200 import reduce_polynomials
    g1 = [(1, (3, 1, 2)), (1, (2, 0, 1))]
    F1 = [[(1, (2, 0, 0)), (1, (0, 1, 0))], [(1, (1, 1, 1)), (1, (0, 0, 1))], [(1, (1, 0, 2)), (1, (0, 2, 0))]]
    g2 = [(1, (5, 10, 4)), (22982, (3, 1, 2))]
    F2 = [[(1, (5, 12, 0)), (25797, (1, 5, 2))], [(1, (1, 3, 1)), (27630, (2, 1, 0))], [(1, (1, 9, 1)), (8749, (2, 0, 0))]]
    rem, steps = reduce_polynomials([[g1], [g2]], [F1, F2])
    assert rem[0][0] == pad8([(1, (0, 1, 2)), (P - 1, (0, 1, 1))])
    assert rem[1][0] == pad8([(2065, (9, 2, 0)), (22982, (3, 1, 2))]) and steps[1][0] == 4
    for (g, F), r, s in zip(((g1, F1), (g2, F2)), rem, steps):
        assert (r[0], s[0]) == orc.reduce(canon(orc, g), [canon(orc, f) for f in F])


# dividends of up to 48 terms against these lists leave remainders of up to ~600 terms in 4 - 5 variables (the oracle's
# reduce), more than the "poly" preset's 512-term scratch holds for the intermediate dividends
ROOMY = dict(max_poly_terms=8192)


def random_case(rng, n, nlists=512, nq=4096, prime=P):
    lists = [[rand_poly(rng, n, int(rng.integers(1, 13)), 3, prime) for _ in range(int(rng.integers(1, 25)))]
             for _ in range(nlists)]
    queries = [rand_poly(rng, n, int(rng.integers(1, 49)), 4, prime) for _ in range(nq)]
    which = rng.integers(0, nlists, size=nq)
    return lists, queries, which


def check_random(torch, orc, eng, n, lists, queries, which, sorted_, prime=P):
    rem, steps, lengths, status = eng.reduce(batch([[q] for q in queries], n, prime), batch(lists, n, prime, True),
                                             which=torch.as_tensor(which), sorted=sorted_)
    assert (status == 2).all(), torch.unique(status, return_counts=True)
    got, steps, lengths = rem.to_lists(), steps.tolist(), lengths.tolist()
    for q, g in enumerate(queries):
        F = [canon(orc, f) for f in lists[which[q]]]
        r, s = orc.reduce(canon(orc, g), by_lead(orc, F) if sorted_ else F)
        assert (pad8(got[q][0]), steps[q], lengths[q]) == (r, s, len(r)), q
    return steps


@pytest.mark.parametrize("sorted_", [False, True])
@pytest.mark.parametrize("n", [3, 5, 6, 8])
def test_random_parity(torch_cuda, orc, n, sorted_):
    rng = np.random.default_rng(1000 * n + sorted_)
    lists, queries, which = random_case(rng, n)
    steps = check_random(torch_cuda, orc, engine(n, **ROOMY), n, lists, queries, which, sorted_)
    assert sum(steps) > len(queries)   # the lists do reduce


def test_scan_order_changes_the_remainder(torch_cuda, orc):
    """F = [xy - z, x - 1], g = xy: in the given order xy - z reduces g to z; sorted by lead monomial x - 1 comes first and
    leaves y.  The oracle agrees in both orders."""
    F = [[(1, (1, 1, 0)), (P - 1, (0, 0, 1))], [(1, (1, 0, 0)), (P - 1, (0, 0, 0))]]
    g = [(1, (1, 1, 0))]
    eng = engine(3, envs=4)
    out = {}
    for s in (False, True):
        rem, steps, _, status = eng.reduce(batch([[g]], 3), batch([F], 3, divisors=True), sorted=s)
        assert status.tolist() == [2]
        out[s] = (pad8(rem[0][0]), steps.tolist()[0])
        Fo = [canon(orc, f) for f in F]
        assert out[s] == orc.reduce(canon(orc, g), by_lead(orc, Fo) if s else Fo)
    assert out[False][0] == pad8([(1, (0, 0, 1))]) and out[True][0] == pad8([(1, (0, 1, 0))])


def test_counters(torch_cuda):
    rng = np.random.default_rng(7)
    lists, queries, which = random_case(rng, 4, nlists=64, nq=512)
    eng = engine(4, envs=256, **ROOMY)
    eng.counters(reset=True)
    _, steps, lengths, status = eng.reduce(batch([[q] for q in queries], 4), batch(lists, 4, divisors=True),
                                           which=torch_cuda.as_tensor(which), return_remainders=False)   # one launch
    assert (status == 2).all(), torch_cuda.unique(status, return_counts=True)
    c = eng.counters()
    assert c["additions"] == int(steps.sum()) and c["term_moves"] == int(lengths.sum())
    assert c["env_steps"] == 0 and c["episodes"] == 0 and c["lms_scanned"] > 0 and c["terms_read"] > 0


@pytest.fixture(scope="module")
def weighted_run(torch_cuda):
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=3552)
    stats, _, out = eng.run_episodes("degree", episodes=16384, return_gb=True, return_basis=True)
    return eng, stats, out


def test_whole_run_bases(torch_cuda, orc, weighted_run):
    """G of every episode reduces to zero by its reduced basis; random polynomials match the oracle on 256 episodes."""
    eng, stats, out = weighted_run
    gb, G = out["gb"], out["basis"]
    done = gb.stored.cpu().numpy()
    assert np.array_equal(done, stats["status"] == 2) and done.any()
    for s in (False, True):
        rem, steps, lengths, status = eng.reduce(G, gb, sorted=s)
        eo = G.ep_offsets.cpu().numpy()
        q_done = np.repeat(done, np.diff(eo))
        st, ln = status.cpu().numpy(), lengths.cpu().numpy()
        assert (st[q_done] == 2).all() and (ln[q_done] == 0).all()
        assert (st[~q_done] == -1).all()
        assert rem.stored.cpu().numpy().tolist() == (G.stored.cpu().numpy() & done).tolist()
    rng = np.random.default_rng(11)
    eps = rng.choice(np.nonzero(done)[0], size=256, replace=False)
    queries = [rand_poly(rng, 3, int(rng.integers(1, 30)), 12) for _ in eps]
    res = [eng.reduce(batch([[q] for q in queries], 3), gb, which=torch_cuda.as_tensor(eps), sorted=s) for s in (False, True)]
    assert res[0][0] == res[1][0] and all(torch_cuda.equal(a, b) for a, b in zip(res[0][1:], res[1][1:]))
    rem, steps = res[0][0].to_lists(), res[0][1].tolist()
    for k, e in enumerate(eps):
        r, s = orc.reduce(canon(orc, queries[k]), [pad8(f) for f in gb[int(e)]])
        assert (pad8(rem[k][0]), steps[k]) == (r, s), int(e)


def test_sympy_normal_forms(torch_cuda):
    sympy = pytest.importorskip("sympy")
    from deepgroebner_b200 import groebner_bases, reduce_polynomials
    rng = np.random.default_rng(5)
    ideals = [[rand_poly(rng, 3, int(rng.integers(2, 4)), 3) for _ in range(int(rng.integers(2, 4)))] for _ in range(60)]
    bases, _ = groebner_bases(ideals)
    queries = [[rand_poly(rng, 3, int(rng.integers(1, 10)), 4)] for _ in ideals]
    rem, _ = reduce_polynomials(queries, bases)
    a, b, c = sympy.symbols("a b c")

    def expr(f):
        return sum(int(co) * a ** e[0] * b ** e[1] * c ** e[2] for co, e in f)

    for G, q, r in zip(bases, queries, rem):
        _, want = sympy.reduced(expr(q[0]), [expr(g) for g in G], a, b, c, modulus=P, order="grevlex")
        terms = sympy.Poly(want, a, b, c, modulus=P).terms(order="grevlex") if want != 0 else []
        assert [(int(co) % P, tuple(m) + (0,) * 5) for m, co in terms] == r[0]


def test_long_polynomials(torch_cuda, orc):
    """cyclic-5's reduced basis and dividends of up to 200 terms: the general merge (warp_merge) path."""
    from deepgroebner_b200 import cyclic, groebner_bases, reduce_polynomials
    bases, _ = groebner_bases([cyclic(5)], capacity="general")
    G = bases[0]
    rng = np.random.default_rng(3)
    queries = [rand_poly(rng, 5, int(rng.integers(100, 201)), 2) for _ in range(64)]
    rem, steps = reduce_polynomials([queries], [G], capacity="general")
    assert max(len(f) for f in G) > 2
    for q, r, s in zip(queries, rem[0], steps[0]):
        assert (r, s) == orc.reduce(canon(orc, q), G)


def test_prime_101(torch_cuda):
    from oracle import oracle as O
    port = O.load_port()
    port.set_prime(101)
    try:
        rng = np.random.default_rng(101)
        lists, queries, which = random_case(rng, 4, nlists=128, nq=1024, prime=101)
        check_random(torch_cuda, port, engine(4, prime=101, envs=256, **ROOMY), 4, lists, queries, which, False, prime=101)
    finally:
        port.set_prime(P)


def test_edge_cases(torch_cuda):
    eng = engine(3, envs=4)
    g = [(7, (2, 1, 0)), (3, (0, 0, 1))]
    F = [[(1, (0, 1, 1)), (2, (1, 0, 0))]]
    rem, steps, lengths, status = eng.reduce(batch([[g], [[]], [g, [(5, (1, 1, 1))]]], 3),
                                             batch([[], F, F + [[(9, (0, 0, 0))]]], 3, divisors=True))
    assert status.tolist() == [2, 2, 2, 2]
    assert rem[0] == [sorted(g, key=lambda t: (-sum(t[1]), t[1][::-1]))] and steps.tolist()[0] == 0   # empty list: g itself
    assert rem[1] == [[]] and steps.tolist()[1] == 0                                                  # zero query
    assert rem[2] == [[], []] and lengths.tolist()[2:] == [0, 0]                                      # a constant empties all


def test_overflow_statuses(torch_cuda):
    eng = engine(3, envs=4, max_basis=4, max_pairs=16, max_terms=16, max_poly_terms=8)
    x = lambda i, j, k: (i, j, k)  # noqa: E731
    big_list = [[(1, x(9, 0, i))] for i in range(5)]                                   # 5 > max_basis
    long_q = [(1, x(0, i, 0)) for i in range(9)]                                       # 9 > max_poly_terms
    full = [[(1, x(20, 0, 0))] + [(1, x(0, 0, i)) for i in range(4)] for _ in range(3)]  # 15 of 16 terms
    short_q = [(1, x(0, 1, 0)), (1, x(0, 0, 2))]                                        # a remainder of 2 terms
    huge_q = [(1, x(40000, 0, 0))]                                                     # above emax
    lists = [big_list, [[(1, x(1, 0, 0))]], full, [[(1, x(1, 0, 0))]]]
    rem, steps, lengths, status = eng.reduce(batch([[short_q], [long_q], [short_q], [huge_q]], 3),
                                             batch(lists, 3, divisors=True))
    assert status.tolist() == [4, 8, 6, 7]   # BASIS, SCRATCH, TERMS, EXPONENT
    assert steps.tolist() == [0] * 4 and lengths.tolist() == [0] * 4
    assert not rem.stored.any() and rem.poly_offsets.tolist() == [0] * 5


def raw(eng, D, q_off, q_ex, q_cf, which, sink=None, counts=None, ptrs=None):
    """bb_reduce with hand-built query tensors; returns (rc, steps, rlen, status) with outputs pre-filled with 77."""
    import torch
    from deepgroebner_b200.buchberger import _ptr, _stream
    dev = eng.device
    nq = which.numel()
    steps, rlen, status = (torch.full((max(nq, 1),), 77, dtype=torch.int32, device=dev) for _ in range(3))
    nl, nqq = counts or (len(D), nq)
    a = [t.to(dev).contiguous() for t in (D.ep_offsets, D.poly_offsets, D.exps, D.coefs, q_off, q_ex, q_cf, which)]
    p = [_ptr(t) for t in a + [steps, rlen, status]]
    for k in ptrs or ():
        p[k] = None
    rc = eng.lib.bb_reduce(eng.h, nl, p[0], p[1], p[2], p[3], nqq, p[4], p[5], p[6], p[7], 0, p[8], p[9], p[10], sink,
                           _stream())
    torch.cuda.synchronize()
    return rc, steps, rlen, status


def test_malformed_and_argument_errors(torch_cuda):
    torch = torch_cuda
    eng = engine(2, envs=4)
    D = batch([[[(1, (1, 0))]], [[(1, (0, 1))]]], 2, divisors=True)
    i64, i32 = torch.int64, torch.int32
    q_off = torch.tensor([0, 2, 4, 6, 7], dtype=i64)
    q_ex = torch.tensor([[0, 1], [2, 0], [2, 0], [0, 1], [2, 0], [0, 1], [1, 1]], dtype=i32)   # query 0 ascending: unsorted
    q_cf = torch.tensor([1, 1, 1, 0, 1, 1, 1], dtype=i32)                                      # query 1 has a zero coefficient
    which = torch.tensor([0, 0, 1, 2], dtype=i32)                                               # query 3: list 2 of 2
    rc, steps, rlen, status = raw(eng, D, q_off, q_ex, q_cf, which)
    assert rc == 0 and status.tolist() == [-1, -1, 2, -1] and rlen.tolist() == [0, 0, 1, 0]
    Dbad = batch([[[(1, (1, 0))]]], 2, divisors=True)
    Dbad.coefs[0] = 32003
    one = (q_off[:2], q_ex[4:6], q_cf[4:6], torch.tensor([0], dtype=i32))   # a valid query: x^2 + y
    assert raw(eng, Dbad, *one)[3].tolist() == [-1]
    Dzero = batch([[[(1, (1, 0))]]], 2, divisors=True)
    Dzero.poly_offsets = torch.tensor([0, 1, 1], dtype=i64, device=Dzero.coefs.device)
    Dzero.ep_offsets = torch.tensor([0, 2], dtype=i64, device=Dzero.coefs.device)   # a zero polynomial in the list
    assert raw(eng, Dzero, *one)[3].tolist() == [-1]
    # argument errors: nothing is launched, the outputs keep their fill
    from deepgroebner_b200 import _lib
    for kw in (dict(counts=(-1, 4)), dict(counts=(2, -1)), dict(ptrs=(0,)), dict(ptrs=(7,)), dict(ptrs=(10,))):
        rc, steps, rlen, status = raw(eng, D, q_off, q_ex, q_cf, which, **kw)
        assert rc < 0 and status.tolist() == [77] * 4 and steps.tolist() == [77] * 4, kw
    for cap, null in ((-1, False), (4, True)):
        t, ref, s = eng._sink(4, 4, 16)
        s.cap_polys = cap
        if null:
            s.lens_dev = None
        rc, _, _, status = raw(eng, D, q_off, q_ex, q_cf, which, sink=C.byref(s))
        assert rc < 0 and status.tolist() == [77] * 4
        assert b"sink" in eng.lib.bb_last_error(eng.h)


def test_tiny_sink(torch_cuda):
    torch = torch_cuda
    rng = np.random.default_rng(9)
    lists, queries, which = random_case(rng, 3, nlists=16, nq=64)
    eng = engine(3, envs=64)
    Pb, Db = batch([[q] for q in queries], 3), batch(lists, 3, divisors=True)
    big = eng.reduce(Pb, Db, which=torch.as_tensor(which))
    small = eng.reduce(Pb, Db, which=torch.as_tensor(which), capacity=(1, 2))
    assert big[0] == small[0] and all(torch.equal(a, b) for a, b in zip(big[1:], small[1:]))
    # the raw call: where = -1 for what did not fit, used[2] counts it, used[0..1] are the exact totals
    from deepgroebner_b200.buchberger import _group_queries
    wq = torch.as_tensor(which, dtype=torch.int32, device=eng.device)
    _, q_off, q_ex, q_cf, wq = _group_queries(Pb.poly_offsets, Pb.exps, Pb.coefs, wq)
    t, ref, s = eng._sink(64, 1, 2)
    rc, steps, rlen, status = raw(eng, Db, q_off, q_ex, q_cf, wq, sink=ref)
    assert rc == 0 and (status == 2).all()
    where, used = t["where"].cpu().numpy(), t["used"].tolist()
    stored = where[:, 0] >= 0
    assert used[0] == 64 and used[1] == int(rlen.sum()) and used[2] == int((~stored).sum()) > 0
    assert stored.sum() <= 1


def test_non_interference(torch_cuda):
    torch = torch_cuda
    from deepgroebner_b200.buchberger import BuchbergerEngine
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=512)
    before, _, out = eng.run_episodes("degree", episodes=2048, return_gb=True)
    rng = np.random.default_rng(4)
    Pb = batch([[rand_poly(rng, 3, 8, 10)] for _ in range(2048)], 3)
    res = []
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in streams:
        with torch.cuda.stream(s):
            res.append(eng.reduce(Pb, out["gb"]))
    torch.cuda.synchronize()
    assert res[0][0] == res[1][0] and all(torch.equal(a, b) for a, b in zip(res[0][1:], res[1][1:]))
    after, _, out2 = eng.run_episodes("degree", episodes=2048, return_gb=True)
    assert before.tobytes() == after.tobytes() and out["gb"] == out2["gb"]
