"""Every episode's reduced Groebner basis and final basis out of a batched run (bb_run_export, run_episodes(return_gb /
return_basis), strat.groebner_bases): the exported polynomials against the episode records' checksums on whole runs, against
the oracle polynomial by polynomial, across runners, batches, pipelines and sink capacities."""
import ctypes as C

import numpy as np
import pytest

from hashing import GOLD2, hash_item, mix64, polys_hash
from helpers import best_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def pad8(G):
    return [[(int(c), tuple(int(x) for x in e) + (0,) * (8 - len(e))) for c, e in g] for g in G]


def _segment_sums(x, offsets):
    with np.errstate(over="ignore"):
        cs = np.concatenate([np.zeros(1, np.uint64), np.cumsum(x, dtype=np.uint64)])
        return cs[offsets[1:]] - cs[offsets[:-1]]


def batch_hashes(b):
    """polys_hash (include/bbenv.h "checksums") of every episode of a PolyBatch, vectorised over the batch."""
    eo, po = b.ep_offsets.cpu().numpy(), b.poly_offsets.cpu().numpy()
    ex = np.zeros((b.exps.shape[0], 8), np.uint64)
    ex[:, :b.exps.shape[1]] = b.exps.cpu().numpy()
    cf = b.coefs.cpu().numpy().astype(np.uint64)
    E = len(eo) - 1
    to = po[eo]
    tl = (np.arange(len(cf)) - np.repeat(to[:-1], np.diff(to))).astype(np.uint64)
    ql = (np.arange(len(po) - 1) - np.repeat(eo[:-1], np.diff(eo))).astype(np.uint64)
    s16, s32, s48, three = np.uint64(16), np.uint64(32), np.uint64(48), np.uint64(3)
    with np.errstate(over="ignore"):
        elo = ex[:, 0] | (ex[:, 1] << s16) | (ex[:, 2] << s32) | (ex[:, 3] << s48)
        ehi = ex[:, 4] | (ex[:, 5] << s16) | (ex[:, 6] << s32) | (ex[:, 7] << s48)
        ht = hash_item(cf, three * tl) + hash_item(elo, three * tl + np.uint64(1)) + hash_item(ehi, three * tl + np.uint64(2))
        hp = mix64(np.diff(po).astype(np.uint64) + GOLD2 * (ql + np.uint64(1)))
        return _segment_sums(ht, to) + _segment_sums(hp, eo) if E else np.zeros(0, np.uint64)


def check_batches(stats, out):
    """Both batches against the records: which episodes are stored, their sizes and their checksums."""
    st = stats["status"]
    for k, (fp, ft, fh, ok) in {"gb": ("gb_polys", "gb_terms", "gb_hash", st == 2),
                                "basis": ("nbasis", "nterms", "basis_hash", (st == 2) | (st == 1))}.items():
        if k not in out:
            continue
        b = out[k]
        assert np.array_equal(b.stored.cpu().numpy(), ok), k
        eo, po = b.ep_offsets.cpu().numpy(), b.poly_offsets.cpu().numpy()
        assert np.array_equal(np.diff(eo), np.where(ok, stats[fp], 0)), k
        assert np.array_equal(np.diff(po[eo]), np.where(ok, stats[ft], 0)), k
        assert np.array_equal(batch_hashes(b)[ok], stats[fh][ok]), k


WHOLE_RUNS = [
    ("3-20-10-weighted", "degree", 16384, 0, 0, 3552),
    ("3-20-10-weighted", "first", 16384, 0, 0, 3552),
    ("3-20-10-weighted", "normal", 16384, 0, 0, 3552),
    ("3-20-10-uniform", "degree", 65536, 0, 0, None),
    ("7-2-5-uniform", "degree", 2048, 3, 0, 1024),
    ("8-3-4-uniform", "normal", 2048, 3, 0, 1024),
    ("cyclic-6", "random", 256, 0, 1234, 256),
]


@pytest.mark.parametrize("dist,strategy,E,seed0,sel_seed0,N", WHOLE_RUNS)
def test_whole_run_every_episode(torch_cuda, dist, strategy, E, seed0, sel_seed0, N):
    """Every episode's exported reduced basis and final basis hash to the record's gb_hash / basis_hash and have its sizes,
    and the records of the run with both sinks attached equal the reference's stored records."""
    from oracle import golden
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    eng = BuchbergerEngine(dist, num_envs=N or resident_envs(0, int(dist.split("-")[0])))
    stats, _, out = eng.run_episodes(strategy, episodes=E, seed_base=seed0, selection_seed=sel_seed0, gamma=0.99,
                                     compute_gb=True, return_gb=True, return_basis=True)
    assert (stats["status"] == 2).all()
    check_batches(stats, out)
    assert golden.mismatches(stats, golden.key(dist, strategy, E, seed0=seed0, sel_seed0=sel_seed0)) == []


def test_polynomials_equal_the_oracle(torch_cuda, port):
    """512 episodes of 3-20-10-weighted: gb[e] == final_gb() and basis[e] == basis() of the oracle's episode, term by term;
    the golden seed-123 episode gives {y, x^2 z^2} under Degree and First."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 512
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=E)
    stats, _, out = eng.run_episodes("degree", episodes=E, return_gb=True, return_basis=True)
    gb, basis = out["gb"].to_lists(), out["basis"].to_lists()
    env = port.env("3-20-10-weighted")
    for e in range(E):
        env.seed(e)
        env.reset()
        env.run(selection="degree")
        assert pad8(gb[e]) == env.final_gb(), e
        assert pad8(basis[e]) == env.basis(), e
    for strategy in ("degree", "first"):
        _, _, out = eng.run_episodes(strategy, episodes=1, seed_base=123, return_gb=True)
        assert out["gb"][0] == [[(1, (0, 1, 0))], [(1, (2, 0, 2))]], strategy


def test_cyclic6_random_polynomials_equal_the_oracle(torch_cuda):
    """32 cyclic-6 episodes under seeded Random selection (k_run_wide): the reduced basis equals the oracle's
    buchberger(F, Random, ..., seed), the final basis equals the oracle env driven through the same pair sequence."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    orc = best_oracle()
    E, sel_seed, cap = 32, 1234, 1 << 14
    eng = BuchbergerEngine("cyclic-6", num_envs=E)
    stats, trace, out = eng.run_episodes("random", episodes=E, selection_seed=sel_seed, trace_episodes=E, trace_cap=cap,
                                         return_gb=True, return_basis=True)
    assert (stats["steps"] <= cap).all()
    gb, basis = out["gb"].to_lists(), out["basis"].to_lists()
    env = orc.env("cyclic-6")
    F, _ = env.reset()
    for e in range(E):
        want, _ = orc.buchberger(F, selection="random", gamma=0.99, seed=sel_seed + e)
        assert pad8(gb[e]) == want, e
        env.reset()
        for i, j in trace[e, :stats["steps"][e], :2]:
            env.step((int(i), int(j)))
        assert pad8(basis[e]) == env.basis(), e


def test_prime_101_coefficients(torch_cuda):
    """At p = 101 the exported coefficients lie in [0, 101) and the polynomials equal the restatement's."""
    from oracle import oracle as O
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 96
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=E, prime=101)
    stats, _, out = eng.run_episodes("normal", episodes=E, seed_base=7, return_gb=True, return_basis=True)
    for k in ("gb", "basis"):
        c = out[k].coefs
        assert int(c.min()) >= 0 and int(c.max()) < 101
    port = O.load_port()
    port.set_prime(101)
    try:
        env = port.env("3-20-10-weighted")
        gb, basis = out["gb"].to_lists(), out["basis"].to_lists()
        for e in range(E):
            env.seed(7 + e)
            env.reset()
            env.run(selection="normal")
            assert pad8(gb[e]) == env.final_gb() and pad8(basis[e]) == env.basis(), e
    finally:
        port.set_prime(32003)


def test_every_runner_exports_the_same(torch_cuda):
    """bb_set_wide modes 0..8 (warp runner, CTA runner and their test configurations) and both preparation modes give
    identical batches on 16 cyclic-6 Random episodes."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 16
    eng = BuchbergerEngine("cyclic-6", num_envs=E)
    runs = []
    for mode in range(9):
        eng.set_wide(mode)
        stats, _, out = eng.run_episodes("random", episodes=E, selection_seed=99, return_gb=True, return_basis=True)
        runs.append((mode, stats, out))
    eng.set_wide(-1)
    for by_warp in (True, False):
        eng.set_prepare_mode(by_warp)
        stats, _, out = eng.run_episodes("random", episodes=E, selection_seed=99, return_gb=True, return_basis=True)
        runs.append(("prepare by_warp=%s" % by_warp, stats, out))
    _, s0, o0 = runs[0]
    check_batches(s0, o0)
    for what, s, o in runs[1:]:
        assert s.tobytes() == s0.tobytes(), what
        assert o["gb"] == o0["gb"] and o["basis"] == o0["basis"], what


def test_two_batches_and_pipelined_calls(torch_cuda):
    """A 70000-episode call (two batches of bb_run) exports what the 65536-episode run followed by a seed_base=65536 run of
    4464 episodes exports; two calls on alternating streams, prepared ahead, with their own sinks export what plain calls do."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    torch = torch_cuda
    E, cut = 70000, 65536
    eng = BuchbergerEngine("3-20-10-uniform", num_envs=2048)
    _, _, whole = eng.run_episodes("degree", episodes=E, return_gb=True, return_basis=True)
    _, _, head = eng.run_episodes("degree", episodes=cut, return_gb=True, return_basis=True)
    _, _, tail = eng.run_episodes("degree", episodes=E - cut, seed_base=cut, return_gb=True, return_basis=True)
    for k in ("gb", "basis"):
        w, h, t = whole[k], head[k], tail[k]
        P, T = int(h.ep_offsets[-1]), int(h.poly_offsets[-1])
        assert torch.equal(w.stored, torch.cat([h.stored, t.stored])), k
        assert torch.equal(w.ep_offsets[:cut + 1], h.ep_offsets) and torch.equal(w.ep_offsets[cut:] - P, t.ep_offsets), k
        assert torch.equal(w.poly_offsets[:P + 1], h.poly_offsets) and torch.equal(w.poly_offsets[P:] - T, t.poly_offsets), k
        assert torch.equal(w.exps, torch.cat([h.exps, t.exps])) and torch.equal(w.coefs, torch.cat([h.coefs, t.coefs])), k

    n = 4096
    plain = [eng.run_episodes("normal", episodes=n, seed_base=b, return_gb=True, return_basis=True) for b in (0, n)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bufs = [torch.empty(n * 72, dtype=torch.uint8, device="cuda") for _ in streams]
    for b, s in zip((0, n), streams):
        with torch.cuda.stream(s):
            eng.prepare_episodes(n, seed_base=b)
    got = []
    for b, s, buf in zip((0, n), streams, bufs):
        with torch.cuda.stream(s):
            got.append(eng.run_episodes("normal", episodes=n, seed_base=b, out=buf, return_gb=True, return_basis=True))
    torch.cuda.synchronize()
    for (s1, _, o1), (s2, _, o2) in zip(plain, got):
        assert s1.tobytes() == s2.tobytes()
        assert o1["gb"] == o2["gb"] and o1["basis"] == o2["basis"]


def _run_export(eng, E, gb=None, basis=None, compute_gb=1, seed_base=0):
    """bb_run_export through ctypes: (rc, records bytes)."""
    from deepgroebner_b200 import _lib
    import torch
    buf = torch.full((E * 72,), 0xAB, dtype=torch.uint8, device="cuda")
    rc = eng.lib.bb_run_export(eng.h, _lib.SELECTION["degree"], E, seed_base, None, 0, 0, 0.99, compute_gb,
                               C.c_void_p(buf.data_ptr()), None, 0, 0, C.c_void_p(torch.cuda.current_stream().cuda_stream),
                               C.byref(gb) if gb is not None else None, C.byref(basis) if basis is not None else None)
    torch.cuda.synchronize()
    return rc, buf.cpu().numpy().tobytes()


def test_small_sink_and_the_repeat(torch_cuda):
    """A sink too small for the run stores exactly the episodes whose where != -1, with the right contents; used[0..1] are
    the totals over every episode that ends done and used[2] counts the ones not stored; the records are byte-identical to
    a run without sinks.  run_episodes with too little room repeats the run and returns the complete result."""
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine
    torch = torch_cuda
    E = 4096
    eng = BuchbergerEngine("5-5-10-uniform", num_envs=1024)
    stats, _, full = eng.run_episodes("degree", episodes=E, return_gb=True)
    want = full["gb"].to_lists()
    rc, plain = _run_export(eng, E)
    assert rc == 0 and plain == stats.tobytes()
    cap_p, cap_t = int(stats["gb_polys"].sum()) // 3, int(stats["gb_terms"].sum()) // 3
    t = dict(lens=torch.zeros(cap_p, dtype=torch.int32, device="cuda"), exps=torch.zeros(cap_t * 5, dtype=torch.int32, device="cuda"),
             coefs=torch.zeros(cap_t, dtype=torch.int32, device="cuda"), where=torch.zeros((E, 2), dtype=torch.int64, device="cuda"),
             used=torch.zeros(3, dtype=torch.int64, device="cuda"))
    sink = _lib.BBPolySink(lens_dev=t["lens"].data_ptr(), exps_dev=t["exps"].data_ptr(), coefs_dev=t["coefs"].data_ptr(),
                           where_dev=t["where"].data_ptr(), used_dev=t["used"].data_ptr(), cap_polys=cap_p, cap_terms=cap_t)
    rc, rec = _run_export(eng, E, gb=sink)
    assert rc == 0 and rec == plain
    where, used = t["where"].cpu().numpy(), t["used"].cpu().tolist()
    stored = where[:, 0] >= 0
    assert 0 < stored.sum() < E
    assert (where[~stored] == -1).all()
    assert used == [int(stats["gb_polys"].sum()), int(stats["gb_terms"].sum()), int((~stored).sum())]
    lens, exps, coefs = t["lens"].cpu().numpy(), t["exps"].cpu().numpy().reshape(-1, 5), t["coefs"].cpu().numpy()
    for e in np.nonzero(stored)[0]:
        p, q = int(where[e, 0]), int(where[e, 1])
        G = []
        for L in lens[p:p + int(stats["gb_polys"][e])]:
            G.append([(int(coefs[q + r]), tuple(int(x) for x in exps[q + r])) for r in range(L)])
            q += int(L)
        assert G == want[e], e
    s2, _, small = eng.run_episodes("degree", episodes=E, return_gb=True, gb_capacity=(10, 10))
    assert s2.tobytes() == stats.tobytes() and small["gb"] == full["gb"]


def test_truncated_and_overflowed_episodes(torch_cuda):
    """max_steps=20: cut episodes (record status running) store no reduced basis and do store their basis.  An episode that
    ends in BB_STATUS_OVERFLOW_BASIS (a handle with a small max_basis) stores neither and its record is unchanged."""
    from deepgroebner_b200.buchberger import BuchbergerEngine
    E = 1024
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=E)
    stats, _, out = eng.run_episodes("degree", episodes=E, max_steps=20, compute_gb=True, return_gb=True, return_basis=True)
    cut = stats["status"] == 1
    assert cut.any() and (stats["status"][~cut] == 2).all()
    check_batches(stats, out)
    assert not out["gb"].stored.cpu().numpy()[cut].any() and out["basis"].stored.cpu().numpy()[cut].all()

    small = BuchbergerEngine("3-20-10-weighted", num_envs=E, max_basis=24)
    plain, _ = small.run_episodes("degree", episodes=E, compute_gb=True)
    stats, _, out = small.run_episodes("degree", episodes=E, compute_gb=True, return_gb=True, return_basis=True)
    assert stats.tobytes() == plain.tobytes()
    over = stats["status"] == 4
    assert over.any()
    check_batches(stats, out)
    assert not out["gb"].stored.cpu().numpy()[over].any() and not out["basis"].stored.cpu().numpy()[over].any()


def test_argument_errors_do_not_launch(torch_cuda):
    """A gb sink with compute_gb = 0, a sink with a NULL buffer and a sink with a negative capacity each fail with a
    message, and the records buffer is left untouched."""
    from deepgroebner_b200 import _lib
    from deepgroebner_b200.buchberger import BuchbergerEngine
    torch = torch_cuda
    E = 64
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=E)
    t = [torch.zeros(4096, dtype=torch.int64, device="cuda") for _ in range(5)]
    good = dict(lens_dev=t[0].data_ptr(), exps_dev=t[1].data_ptr(), coefs_dev=t[2].data_ptr(), where_dev=t[3].data_ptr(),
                used_dev=t[4].data_ptr(), cap_polys=1000, cap_terms=1000)
    cases = [(dict(good), dict(gb=True, compute_gb=0), b"compute_gb"),
             (dict(good, exps_dev=None), dict(gb=True), b"NULL"),
             (dict(good, where_dev=None), dict(basis=True), b"NULL"),
             (dict(good, cap_terms=-1), dict(basis=True), b"negative"),
             (dict(good, cap_polys=-5), dict(gb=True), b"negative")]
    for fields, how, msg in cases:
        sink = _lib.BBPolySink(**fields)
        rc, rec = _run_export(eng, E, gb=sink if how.get("gb") else None, basis=sink if how.get("basis") else None,
                              compute_gb=how.get("compute_gb", 1))
        assert rc < 0 and msg in eng.lib.bb_last_error(eng.h), (fields, how)
        assert rec == b"\xab" * (E * 72)
        assert all(int(x.abs().sum()) == 0 for x in t)


def test_groebner_bases_known_answers(torch_cuda):
    """tests/test_buchberger.py:236, 239 of the reference: the twisted cubic and cyclic-3 under every elimination."""
    from deepgroebner_b200 import groebner_bases
    from deepgroebner_b200.strat import parse_ideal_string
    orc = best_oracle()
    p = 32003
    x = lambda a, b, c: (a, b, c, 0, 0, 0, 0, 0)
    cubic = parse_ideal_string("b-a^2|c-a^3")
    cyclic3 = parse_ideal_string("a+b+c|a*b+b*c+c*a|a*b*c-1")
    for elim in ("none", "lcm", "gebauermoeller"):
        bases, stats = groebner_bases([cubic, cyclic3], elimination=elim)
        assert bases[0] == [[(1, x(0, 2, 0)), (p - 1, x(1, 0, 1))], [(1, x(1, 1, 0)), (p - 1, x(0, 0, 1))],
                            [(1, x(2, 0, 0)), (p - 1, x(0, 1, 0))]], elim
        assert len(bases[1]) == 3, elim
        for F, G in zip((cubic, cyclic3), bases):
            assert G == orc.buchberger(F, elimination=elim)[0], elim


def test_groebner_bases_of_an_ideal_file(torch_cuda, tmp_path):
    """1000 random 3-20-10-weighted ideals, written with write_ideal_file and read back: every basis equals the oracle's
    buchberger(F)[0]; the statistics equal strategy_stats'."""
    from deepgroebner_b200.strat import groebner_bases, read_ideal_file, strategy_stats, write_ideal_file
    orc = best_oracle()
    gen = orc.generator("3-20-10-weighted")
    gen.seed(4242)
    path = str(tmp_path / "ideals.csv")
    write_ideal_file(path, [gen.next() for _ in range(1000)])
    ideals = read_ideal_file(path)
    bases, stats = groebner_bases(ideals)
    for i, F in enumerate(ideals):
        assert bases[i] == orc.buchberger(F)[0], i
    z, nz, adds = strategy_stats(ideals, "degree")
    assert np.array_equal(z, stats["zero_reductions"]) and np.array_equal(nz, stats["nonzero_reductions"])
    assert np.array_equal(adds, stats["additions"])
    out = str(tmp_path / "bases.csv")
    write_ideal_file(out, bases)
    assert read_ideal_file(out) == bases
